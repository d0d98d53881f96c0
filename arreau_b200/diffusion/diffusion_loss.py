"""Mirror of diffusion/diffusion_loss.py: DiffusionLoss.predict_scores / sample with the reference's
signatures.  The sampler keeps the whole state on the GPU and runs each step as one C call
(arreau_denoise_step); the reference's torch CPU RNG stream (angles via numpy, randn lengths, randn frac, then
per step randn_like(lengths), randn_like(frac), rand((N,Z)) -- SURVEY 3.1) is drawn on the host exactly as the
reference draws it unless `device_noise=True` asks for the in-kernel Philox generator, or `crystal_ids` asks for draws
keyed per crystal on the device (initial state and step noise), which make a crystal's trajectory independent of the
batch it is sampled in."""
from __future__ import annotations

from typing import Optional

import attr
import numpy as np
import torch
import torch.nn.functional as F

from .. import _lib
from ..engine import DenoiseEngine, allowed_state_words, known_lattices, known_rows
from ..tables import POS_SIGMA_MAX, POS_SIGMA_MIN, build_tables
from .d3pm import D3PM
from .diffusion_helpers import VE_pbc, VP_lattice
from .lattice_helpers import matrix_to_params

pos_sigma_min = POS_SIGMA_MIN
pos_sigma_max = POS_SIGMA_MAX


@attr.s(auto_attribs=True, frozen=True)
class SampleResult:
    """diffusion/diffusion_loss.py:39-49."""
    frac_x: np.ndarray = None
    atomic_numbers: np.ndarray = None
    lattice: np.ndarray = None
    idx_start: np.ndarray = None
    num_atoms: np.ndarray = None


def sample_bravais_angles(lattice_type: str = "monoclinic"):
    """diffusion/diffusion_helpers.py:739-774, monoclinic branch (:752-755): degrees, consumed as radians (B5)."""
    if lattice_type != "monoclinic":
        raise NotImplementedError(lattice_type)
    return [90.0, np.random.uniform(90, 180), 90.0]


def _fourier_w(t_emb_weights):
    """The Gaussian Fourier frequencies of a GaussianFourierProjection, or the frequencies themselves."""
    return getattr(t_emb_weights, "gaussian_fourier_proj_w", t_emb_weights)


class _TrainStepLoss(torch.autograd.Function):
    """The scalar loss of one training step as an autograd node: the step's kernels have already produced the flat
    gradient buffer (TrainEngine.loss_and_grads), backward() hands its slices to the parameters."""

    @staticmethod
    def forward(ctx, engine, names, out_dtype, *params):
        ctx.engine, ctx.names = engine, names
        return engine.loss[0].to(out_dtype).clone()

    @staticmethod
    def backward(ctx, grad_out):
        gv = ctx.engine.p.grad_views()
        scale = grad_out.to(torch.float32)
        return (None, None, None) + tuple(gv[n] * scale for n in ctx.names)


class DiffusionLoss(torch.nn.Module):
    """diffusion/diffusion_loss.py:67-93.  `args` needs .radius, .max_neighbors, .num_timesteps."""

    def __init__(self, args, num_atomic_states: int, precision: str = "fp32"):
        super().__init__()
        self.cutoff, self.max_neighbors, self.T = args.radius, args.max_neighbors, args.num_timesteps
        self.num_atomic_states = num_atomic_states
        self.precision = precision
        self.tables = build_tables(self.T, num_atomic_states)
        self.pos_diffusion = VE_pbc(self.T, sigma_min=pos_sigma_min, sigma_max=pos_sigma_max)
        self.d3pm = D3PM(x0_model=None, n_T=self.T, num_classes=num_atomic_states, forward_type="mask")
        self.lattice_diffusion = VP_lattice(num_steps=self.T)
        self._engine = None
        self._engine_key = None
        self._train_engines = {}
        self._eval_engines = {}
        self.backward_precision = "fp32"      # "tf32": tensor-core GEMMs in the backward pass (training.py)
        self.coord_loss_weight = self.atom_type_loss_weight = self.lattice_loss_weight = 1

    @staticmethod
    def _same_device(have, want) -> bool:
        """torch.device("cuda") names the current device: it must compare equal to the "cuda:0" a tensor reports."""
        have, want = torch.device(have), torch.device(want)
        if have.type != want.type:
            return False
        if have.type != "cuda" or have.index == want.index:
            return True
        if have.index is not None and want.index is not None:
            return False
        cur = torch.cuda.current_device()
        return (cur if have.index is None else have.index) == (cur if want.index is None else want.index)

    # -- engine cache: one per (model weights, topology) --------------------------------------------
    def packed_weights(self, net, device):
        """The kernel layouts of net's current weights.  Engines read a packed COPY of the weights: a training step /
        load_state_dict / callibrate in between bumps the version of the flat parameter buffer, and the copy is rebuilt
        (ADVICE r1: sample -> train -> sample must not sample from the pre-training weights)."""
        version = (getattr(getattr(net, "flat", None), "version", 0), getattr(net, "_pack_epoch", 0))
        if getattr(net, "_packed", None) is None or getattr(net, "_packed_version", None) != version \
                or not self._same_device(net._packed.device, device):
            net.pack(device)
            net._packed_version = version
        return net._packed

    def engine_for(self, model, t_emb_weights, num_atoms, device, debug=False) -> DenoiseEngine:
        net = getattr(model, "model", model)          # PONITA_DIFFUSION.model or a bare PonitaFiberBundle
        na = tuple(int(v) for v in torch.as_tensor(num_atoms).reshape(-1).tolist())
        key = (id(net), na, str(device), debug, self.precision)
        packed = self.packed_weights(net, device)
        if self._engine is None or self._engine_key != key:
            self._engine = DenoiseEngine(packed, self.tables, _fourier_w(t_emb_weights), na, self.cutoff,
                                         self.max_neighbors, precision=self.precision, debug=debug, device=device)
            self._engine_key = key
        elif self._engine.w is not packed:
            self._engine.w = packed
        return self._engine

    @staticmethod
    def _batch_engine(cache: dict, key, num_atoms, build, capacity=None, headroom: float = 1.25):
        """The capacity-based engine cache[key], re-bound to the batch topology `num_atoms`.  It is rebuilt by
        build(node_capacity, crystal_capacity) only when there is none or the batch exceeds its capacity: for
        `capacity` (atoms, crystals), by default `headroom` x this batch, never below the old engine's."""
        eng = cache.get(key)
        if eng is not None and eng.fits(num_atoms):
            if tuple(num_atoms) != eng.eng.topology:
                eng.set_topology(num_atoms)
            return eng
        n_cap, g_cap = capacity or (int(sum(num_atoms) * headroom), int(len(num_atoms) * headroom))
        if eng is not None:
            n_cap, g_cap = max(n_cap, eng.eng.N_cap), max(g_cap, eng.eng.G_cap)
        cache.pop(key, None)
        eng = None                                          # free the old buffers before allocating the larger ones
        cache[key] = eng = build(n_cap, g_cap)
        return eng

    # -- training step (diffusion_loss.py:95-110,199-274) ---------------------------------------------
    def train_engine_for(self, net, t_emb_weights, num_atoms, device):
        """ONE capacity-based TrainEngine per (parameters, backward precision): every batch topology (atoms per crystal)
        is bound to its buffers in place; it is rebuilt -- with headroom -- only when a batch exceeds the capacity
        (the first batches of the first epoch), so a shuffled epoch does not reallocate (`self.train_engine_builds`
        counts the builds)."""
        from ..training import TrainEngine
        flat = net.flat if getattr(net, "flat", None) is not None and self._same_device(net.flat.device, device) \
            else net.flatten_parameters(device)
        na = [int(v) for v in torch.as_tensor(num_atoms).reshape(-1).tolist()]

        def build(n_cap, g_cap):
            te = TrainEngine(flat, self.tables, _fourier_w(t_emb_weights), net.ori_grid, na, self.cutoff,
                             self.max_neighbors, device=device, backward_precision=self.backward_precision,
                             node_capacity=n_cap, crystal_capacity=g_cap)
            self.train_engine_builds = getattr(self, "train_engine_builds", 0) + 1
            return te
        return self._batch_engine(self._train_engines, (id(flat), self.backward_precision), na, build)

    # -- evaluation (validation / test loss, arreau_b200/evaluation.py) --------------------------------
    def eval_engine_for(self, net, t_emb_weights, num_atoms, device, capacity=None):
        """ONE capacity-based EvalEngine (model precision, its own buffers: the training and sampling engines are not
        touched), re-bound to every batch topology; rebuilt only when a batch exceeds the capacity, and dropped when
        the precision or the device changes.  capacity: (atoms, crystals) to size it for up front."""
        from ..evaluation import EvalEngine
        na = [int(v) for v in np.asarray(num_atoms).reshape(-1)]
        key = (self.precision, torch.device(device))
        if key not in self._eval_engines:
            self._eval_engines.clear()                      # one evaluation engine
        build = lambda n_cap, g_cap: EvalEngine(  # noqa: E731
            self.packed_weights(net, device), self.tables, _fourier_w(t_emb_weights), na, self.cutoff, self.max_neighbors,
            precision=self.precision, device=device, node_capacity=n_cap, crystal_capacity=g_cap)
        return self._batch_engine(self._eval_engines, key, na, build, capacity)

    @torch.no_grad()
    def evaluate(self, model, batch, t_emb_weights, crystal_ids, seed: int = 0, timestep=None, noise=None,
                 capacity=None):
        """Forward-only loss of a batch, per crystal (no backward, no torch RNG, the training state untouched):
        returns an EvalResult (t[G], num_atoms[G], terms[G,4]; see arreau_b200/evaluation.py).  The draws are keyed by
        (seed, crystal_ids[g]) (arreau_eval_noise), so a crystal's terms do not depend on the batch it is in;
        `timestep` / `noise` inject draws as in __call__.  Precision: self.precision."""
        from ..evaluation import EvalResult
        dev = batch.X0.device
        if dev.type != "cuda":
            raise RuntimeError("arreau_b200 runs on CUDA tensors only (no CPU fallback)")
        net = getattr(model, "model", model)
        na = getattr(batch, "num_atoms_cpu", None)
        na = np.asarray(batch.num_atoms.cpu() if na is None else na, dtype=np.int64)
        ee = self.eval_engine_for(net, t_emb_weights, na, dev, capacity=capacity)
        ee.eng.w = self.packed_weights(net, dev)
        t, terms = ee.run(batch.X0, batch.A0, batch.L0.view(-1, 3, 3), crystal_ids, seed, timestep, noise)
        return EvalResult(t=t.clone(), num_atoms=torch.from_numpy(na.copy()), terms=terms.clone())

    def compute_frac_x_error(self, pred_frac_eps_x, target_frac_eps_x, batch=None):
        """diffusion_loss.py:95-110 (value only; gradients flow through __call__)."""
        d = torch.clamp(torch.remainder((pred_frac_eps_x - target_frac_eps_x).abs(), 1), min=0, max=1)
        d = torch.min(d, 1 - d)
        return torch.mean(torch.sum(d ** 2, dim=1))

    def diffuse_lattice_params(self, lattice: torch.Tensor, t_int: torch.Tensor):
        """diffusion_loss.py:199-202."""
        lengths, angles = matrix_to_params(lattice)
        noisy_lengths, _ = self.lattice_diffusion(lengths, t_int)
        return noisy_lengths, lengths, angles

    def __call__(self, model, batch, t_emb_weights, timestep=None, noise=None):
        """diffusion_loss.py:204-274: samples t and the noise (the reference's draws, in its order, on the batch's
        device), noises the batch, predicts, and returns the scalar loss.  The returned tensor is attached to the
        model's parameters: `.backward()` delivers the gradients the step's backward kernels produced.  `noise`
        optionally injects (eps_x[N,3], u[N,Z], eps_l[G,3]).  Loss parts of the last call: `self.last_loss_parts`."""
        frac_x_0, atom_type_0 = batch.X0, batch.A0
        lattice_0 = batch.L0.view(-1, 3, 3)
        num_atoms = batch.num_atoms
        dev = frac_x_0.device
        if dev.type != "cuda":
            raise RuntimeError("arreau_b200 runs on CUDA tensors only (no CPU fallback)")
        G, N, Z = num_atoms.size(0), frac_x_0.shape[0], self.num_atomic_states
        if timestep is None:
            timestep = torch.randint(1, self.T + 1, size=(G, 1), device=dev).long()
        else:
            timestep = torch.ones((G, 1), device=dev).long() * timestep
        if noise is None:   # VE_pbc.forward, D3PM.get_xt, VP_lattice.forward draw in this order (:228-237)
            eps_x = torch.randn_like(frac_x_0)
            u = torch.rand((N, Z), device=dev)
            eps_l = torch.randn((G, 3), device=dev, dtype=frac_x_0.dtype)
        else:
            eps_x, u, eps_l = noise
        net = getattr(model, "model", model)
        # the batch topology from the host copy when the collate left one (no device -> host read per step)
        te = self.train_engine_for(net, t_emb_weights, getattr(batch, "num_atoms_cpu", num_atoms), dev)
        te.loss_and_grads(frac_x_0, atom_type_0, lattice_0, timestep, eps_x, u, eps_l)
        self.last_loss_parts = te.loss
        names = [n for n, p in net.named_parameters() if p.numel() > 0]
        params = [p for _, p in net.named_parameters() if p.numel() > 0]
        return _TrainStepLoss.apply(te, names, frac_x_0.dtype, *params)

    forward = __call__

    def predict_scores(self, noisy_frac_x, noisy_atom_types, t_feat, num_atoms, noisy_lengths, angles, model, batch,
                       t_emb_weights):
        """diffusion/diffusion_loss.py:112-197.  noisy_atom_types is the one-hot [N,Z] of the reference."""
        dev = noisy_frac_x.device
        if dev.type != "cuda":
            raise RuntimeError("arreau_b200 runs on CUDA tensors only (no CPU fallback)")
        eng = self.engine_for(model, t_emb_weights, num_atoms, dev)
        types = noisy_atom_types.argmax(-1) if noisy_atom_types.dim() == 2 else noisy_atom_types
        eng.set_state(noisy_frac_x, types, noisy_lengths, angles)
        tt = t_feat.reshape(-1)
        score, logits, len0 = eng.predict_scores(tt)
        dt = noisy_frac_x.dtype
        return score.to(dt).clone(), logits.to(dt).clone(), len0.to(dt).clone()

    @torch.no_grad()
    def sample(self, *, model, z_table, t_emb_weights, num_atoms_per_sample: int, num_samples_in_batch: int,
               vis_name: str = "", visualization_setting=None, show_bonds: bool = False,
               constant_atoms: Optional[torch.Tensor] = None, num_atoms: Optional[torch.Tensor] = None,
               device="cuda", device_noise: bool = False, seed: int = 0, step_callback=None,
               cuda_graph: bool = False, crystal_ids=None, allowed_states=None, initial_types=None,
               known_frac=None, known_lattice=None) -> SampleResult:
        """diffusion/diffusion_loss.py:277-377.  Extra keyword-only options (defaults reproduce the reference):
        `num_atoms` a per-crystal atom-count vector, `device_noise` Philox noise generated on the GPU,
        `step_callback(timestep, engine)` called after each step (e.g. to log E/N), `cuda_graph` (needs device_noise or
        crystal_ids, and max_neighbors > 0): the loop body is captured once and replayed T - 1 times, one launch per
        step -- bit-identical results; it pays for small batches, whose steps are launch bound.
        `crystal_ids` (G integers): the initial state and every step's noise are drawn on the device per crystal, keyed
        by (seed, id) (arreau_sample_init_keyed / arreau_sample_noise_keyed), so a crystal's trajectory depends on the
        weights, the precision, the seed, its id and its atom count only -- not on the batch it is sampled in.  The
        host generators (numpy, torch) are not touched; device_noise is implied.
        `allowed_states` (bool [G,Z], or [Z] for every crystal): the states each crystal's atoms may take -- the type
        update samples from the model's x0 prediction restricted to them (arreau_d3pm_reverse_allowed); leave the mask
        state Z-1 out and every atom ends on an allowed element.  It cannot be combined with constant_atoms.
        `initial_types` (N states): the atoms' initial states instead of the mask state Z-1; unlike constant_atoms they
        are then updated like any state.  Used for the types of known atoms.
        `known_frac` ([N,3], NaN rows for free atoms) and `known_lattice` ([G,3,3], NaN matrices for free crystals):
        structure-conditioned sampling (DenoiseEngine.set_known): the known positions, with the known atoms' initial
        states as their types, and the known lattices are imposed on every step by replacement, and are the final
        state's.  A known atom needs a type: its initial state may not be the mask state.  A known lattice needs
        |det| >= 0.1 A^3."""
        Z = len(z_table)
        G = num_samples_in_batch
        na = torch.full((G,), num_atoms_per_sample) if num_atoms is None else torch.as_tensor(num_atoms).reshape(-1)
        N = int(na.sum())
        if allowed_states is not None:         # checked before any device work
            if constant_atoms is not None:
                raise ValueError("allowed_states restricts the type update, which constant_atoms switches off")
            allowed_state_words(allowed_states, G, Z)
        if initial_types is not None:
            if constant_atoms is not None:
                raise ValueError("initial_types and constant_atoms exclude each other")
            initial_types = torch.as_tensor(initial_types).reshape(-1).to(torch.int64)
            if initial_types.shape[0] != N or bool(((initial_types < 0) | (initial_types >= Z)).any()):
                raise ValueError(f"initial_types must hold {N} states in 0..{Z - 1}")
        atom_types = (constant_atoms if constant_atoms is not None else
                      initial_types if initial_types is not None else torch.full((N,), Z - 1))
        if known_frac is not None:
            _, known = known_rows(known_frac, (N, 3), "known frac")
            untyped = torch.nonzero(known & (torch.as_tensor(atom_types).reshape(-1) == Z - 1)).reshape(-1)
            if untyped.numel():
                raise ValueError(f"known atom {int(untyped[0])} has no type (its initial state is the mask state)")
        if known_lattice is not None:
            known_lattices(known_lattice, G)
        dd = torch.float64                                     # main_diffusion_generate.py:27
        keyed = crystal_ids is not None
        if keyed:
            crystal_ids = torch.as_tensor(crystal_ids).reshape(-1)
            if crystal_ids.shape[0] != G:
                raise ValueError(f"{crystal_ids.shape[0]} crystal ids for {G} crystals")
        else:
            angles = torch.tensor([sample_bravais_angles("monoclinic") for _ in range(G)], dtype=dd)
            lengths = torch.randn([G, 3], dtype=dd)
        if not keyed:
            frac_x = torch.randn([N, 3], dtype=dd) * pos_sigma_max
        eng = self.engine_for(model, t_emb_weights, na, torch.device(device))
        eng.set_allowed_states(allowed_states)
        if keyed:
            eng.set_crystal_ids(crystal_ids)
            eng.init_state_keyed(seed, atom_types, pos_sigma_max)
        else:
            eng.set_state(frac_x, atom_types, lengths, angles)
        eng.set_known(known_frac, known_lattice)      # after the state: it overrides the known lattices' drawn angles
        if cuda_graph and (not (device_noise or keyed) or self.max_neighbors <= 0):
            raise ValueError("cuda_graph=True needs device_noise=True (or crystal_ids) and max_neighbors > 0")
        if cuda_graph:
            g = eng.capture_trajectory_graph(self.T - 1, seed, update_types=constant_atoms is None, keyed=keyed)
            for timestep in reversed(range(1, self.T)):
                g.replay()
                if step_callback is not None:
                    step_callback(timestep, eng)
        for step_idx, timestep in enumerate(reversed(range(1, self.T)) if not cuda_graph else ()):
            if keyed:
                eng.draw_noise_keyed(seed, step_idx)
            elif device_noise:
                eng.draw_noise(seed, step_idx)
            else:   # the reference's draw order per step: lengths, frac, types
                eng.set_noise(torch.randn(G, 3, dtype=dd), torch.randn(N, 3, dtype=dd), torch.rand(N, Z, dtype=dd))
            eng.step(timestep, update_types=constant_atoms is None)
            if step_callback is not None:
                step_callback(timestep, eng)
        types = eng.types.cpu()
        zs = np.asarray(z_table.zs if hasattr(z_table, "zs") else z_table)
        return SampleResult(num_atoms=na.numpy(), frac_x=eng.frac.cpu().numpy(), atomic_numbers=zs[types.numpy()],
                            lattice=eng.lattice.cpu().numpy())
