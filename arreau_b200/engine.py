"""DenoiseEngine: device buffers + launch sequences of the denoising step.

Host logic only (buffer ownership, argument structs, the sampler loop); every computation is a kernel
of libarreau_b200.so reached through arreau_b200._lib.  One engine = one batch topology (num_atoms per
crystal) on one GPU.  Mirrors the loop body of DiffusionLoss.sample (diffusion/diffusion_loss.py:318-349).
"""
from __future__ import annotations

import ctypes as C
from typing import Optional, Sequence, Tuple

import numpy as np
import torch

from . import _lib
from .tables import DiffusionTables
from .weights import HIDDEN, LAYERS, NUM_ORI, PonitaWeights

PRECISIONS = {"fp32": _lib.PRECISION_FP32, "fp16": _lib.PRECISION_FP16}


def angle_factors(angles: torch.Tensor) -> torch.Tensor:
    """[sin b, cos b, sin a, cos g*, sin g*, cos a] per crystal with the reference's own torch expressions
    (diffusion/lattice_helpers.py:76-82).  The angles are constants of a sampling trajectory
    (diffusion_loss.py:294-296), so this runs once per set_state on the host like the schedule tables; the
    per-step lattice is then pure fp64 products on the device (arreau_lattice_from_trig) and bit-identical to
    the reference's, which keeps exact-tie neighbour selection in degenerate cells identical too."""
    alpha, beta, gamma = angles.unbind(-1)
    cos_a, cos_b, cos_g = torch.cos(alpha), torch.cos(beta), torch.cos(gamma)
    sin_a, sin_b = torch.sin(alpha), torch.sin(beta)
    val = torch.clamp((cos_a * cos_b - cos_g) / (sin_a * sin_b), -1.0, 1.0)
    gs = torch.arccos(val)
    return torch.stack([sin_b, cos_b, sin_a, torch.cos(gs), torch.sin(gs), cos_a], dim=1)


def _i32(a, device):
    return torch.as_tensor(np.asarray(a), dtype=torch.int32).to(device)


class DenoiseEngine:
    """Buffers are sized once for a CAPACITY (atoms, crystals, edges) and a batch topology (atoms per crystal) is bound
    to them in place with `set_topology`: every kernel takes N / G as arguments and bounds itself, so shuffled
    variable-size batches (training, SURVEY 8f-4) re-use one engine without reallocating.  By default the capacity
    is the topology given to the constructor."""

    # per-atom / per-crystal buffers: name -> (leading extent kind, trailing shape, dtype)
    _NODE_BUFS = {"frac": ((3,), torch.float64), "types": ((), torch.int64), "pos": ((3,), torch.float64),
                  "raw_count": ((), torch.int32), "deg": ((), torch.int32), "crystal_of_atom": ((), torch.int32),
                  "t_of_atom": ((), torch.int32), "vec": ((4, 3), torch.float32), "score": ((3,), torch.float32),
                  "h": ((NUM_ORI, HIDDEN), torch.float32), "x1": ((NUM_ORI, HIDDEN), torch.float32),
                  "z_frac": ((3,), torch.float64)}
    _CRYSTAL_BUFS = {"lengths": ((3,), torch.float64), "angles": ((3,), torch.float64), "lattice": ((3, 3), torch.float64),
                     "angle_trig": ((6,), torch.float64), "num_neighbors_image": ((), torch.int64),
                     "len0": ((3,), torch.float32), "z_len": ((3,), torch.float64), "num_atoms": ((), torch.int64),
                     "crystal_id": ((), torch.int64)}

    def __init__(self, weights: PonitaWeights, tables: DiffusionTables, fourier_w, num_atoms: Sequence[int],
                 radius: float, max_neighbors: int, precision: str = "fp32", edge_capacity: Optional[int] = None,
                 debug: bool = False, device="cuda", pooled_readout: bool = True,
                 node_capacity: Optional[int] = None, crystal_capacity: Optional[int] = None):
        if precision not in PRECISIONS:
            raise ValueError(f"precision must be one of {sorted(PRECISIONS)}")
        _lib.load()
        self.w, self.tabs = weights, tables
        self.device = torch.device(device)
        self.precision, self.debug = precision, debug
        self.radius, self.cap = float(radius), int(max_neighbors)
        na = np.asarray(num_atoms, dtype=np.int64).reshape(-1)
        self.Z = weights.num_states
        if tables.Z != self.Z:
            raise ValueError(f"tables built for {tables.Z} atom states, weights have {self.Z}")
        dev = self.device
        Z = self.Z
        self.N_cap = max(int(na.sum()), int(node_capacity or 0), 1)
        self.G_cap = max(int(na.shape[0]), int(crystal_capacity or 0), 1)
        Nc, Gc = self.N_cap, self.G_cap
        self.F = weights.num_scalar
        self.emb = (self.F - Z - 10) // 2
        self._bufs = {}
        z = lambda shape, dt: torch.zeros(shape, dtype=dt, device=dev)  # noqa: E731
        for name, (tail, dt) in self._NODE_BUFS.items():
            self._bufs[name] = ("N", z((Nc,) + tail, dt))
        for name, (tail, dt) in self._CRYSTAL_BUFS.items():
            self._bufs[name] = ("G", z((Gc,) + tail, dt))
        self._bufs["x"] = ("N", z((Nc, self.F), torch.float32))
        self._bufs["logits"] = ("N", z((Nc, Z), torch.float32))
        self._bufs["acc"] = ("N", z((Nc, Z + 6), torch.float32))
        self._bufs["u_type"] = ("N", z((Nc, Z), torch.float64))
        self._bufs["row_ptr"] = ("N+1", z((Nc + 1,), torch.int32))
        self._bufs["atom_offset"] = ("G+1", z((Gc + 1,), torch.int32))
        self.overflow_flag = z((1,), torch.int32)
        # orientation-pooled features per layer: the fp16 path's read-outs run on these (arreau_readout_pooled)
        # (arreau_readout_pooled is specialised on Z + 6 == 96 output columns, i.e. the reference's 90 atom states;
        # any other z_table takes the per-layer read-out arreau_readout_accumulate, Z <= 100)
        self._pool_flat = (z(((LAYERS + 1) * ((Nc + 15) // 16) * 4 * HIDDEN * 16,), torch.float32)
                           if (self.precision == "fp16" and pooled_readout and "readout_v" in weights.t and Z + 6 == 96)
                           else None)
        if precision == "fp16":     # 128-row UMMA tile images (32 KB each), see arreau_message_fiber_norm
            self.y = torch.zeros(((Nc * NUM_ORI + 127) // 128) * 128 * HIDDEN, device=dev, dtype=torch.float16)
        else:
            self.y = torch.zeros(Nc * NUM_ORI * HIDDEN, device=dev, dtype=torch.float32)
        # tables
        self.d_vp_betas = tables.vp_betas.to(torch.float64).to(dev)
        self.d_ve_sigmas = tables.ve_sigmas.to(torch.float64).to(dev)
        self.d_q_keep, self.d_q_to_mask = tables.q_keep.to(dev), tables.q_to_mask.to(dev)
        self.d_fourier_w = torch.as_tensor(np.asarray(fourier_w.detach().cpu() if isinstance(fourier_w, torch.Tensor)
                                                      else fourier_w), dtype=torch.float64).to(dev)
        if self.d_fourier_w.numel() != self.emb:
            raise ValueError(f"time embedding has {self.d_fourier_w.numel()} frequencies, the model expects {self.emb}")
        self.edge_capacity = -1
        self.G = self.N = 0
        self._debug_flat = None
        self._alloc_edges(int(edge_capacity) if edge_capacity is not None else
                          (Nc * self.cap if self.cap > 0 else max(1, 32 * Nc)))
        self.set_topology(na)

    # ------------------------------------------------------------------ topology
    def set_topology(self, num_atoms: Sequence[int]) -> None:
        """Bind a batch topology (atoms per crystal) to the preallocated buffers: index arrays are rewritten in place,
        the public tensors (`frac`, `types`, `h`, `logits`, ...) become views of the first N / G rows, the argument
        structs get the new extents.  No allocation; raises if the batch exceeds the capacity."""
        na = np.asarray(num_atoms, dtype=np.int64).reshape(-1)
        G, N = int(na.shape[0]), int(na.sum())
        if N > self.N_cap or G > self.G_cap:
            raise ValueError(f"batch of {N} atoms / {G} crystals exceeds the engine capacity {self.N_cap} / {self.G_cap}")
        if self.cap > 0 and N * self.cap > self._edge_alloc:
            raise ValueError("edge capacity too small for this batch")
        self.G, self.N = G, N
        # capped graphs: E <= N * cap for THIS batch; kernels that walk "capacity" rows (the training backward) and the
        # layer stride of the kernel slab follow the bound batch, not the allocation
        self._bind_edges(N * self.cap if self.cap > 0 else self._edge_alloc)
        self.topology = tuple(int(v) for v in na)
        off = np.zeros(G + 1, dtype=np.int64)
        np.cumsum(na, out=off[1:])
        ext = {"N": N, "G": G, "N+1": N + 1, "G+1": G + 1}
        for name, (kind, buf) in self._bufs.items():
            setattr(self, name, buf[: ext[kind]])
        # pinned staging + non_blocking: a plain copy_ from pageable memory synchronises the stream, i.e. a training loop
        # that binds a new topology every step would drain the GPU before enqueueing the next step (the caching host
        # allocator keeps a staging block alive until its copy has run)
        stage = (lambda a: torch.as_tensor(a).pin_memory()) if self.device.type == "cuda" else torch.as_tensor
        self.atom_offset.copy_(stage(off.astype(np.int32)), non_blocking=True)
        self.crystal_of_atom.copy_(stage(np.repeat(np.arange(G), na).astype(np.int32)), non_blocking=True)
        self.num_atoms.copy_(stage(na), non_blocking=True)
        groups = (N + 15) // 16
        self.pool = (self._pool_flat[: (LAYERS + 1) * groups * 4 * HIDDEN * 16].view(LAYERS + 1, groups, 4, HIDDEN, 16)
                     if self._pool_flat is not None else None)
        if self._debug_flat is not None:
            node = N * NUM_ORI * HIDDEN
            d = self._debug_flat
            self.x1_debug = d[0][: LAYERS * node].view(LAYERS, N, NUM_ORI, HIDDEN)
            self.x2_debug = d[1][: LAYERS * node].view(LAYERS, N, NUM_ORI, HIDDEN)
            self.h_debug = d[2][: (LAYERS + 1) * node].view(LAYERS + 1, N, NUM_ORI, HIDDEN)
        if hasattr(self, "_noise_sets"):      # staged-noise double buffers are bound to the old extents
            del self._noise_sets
        self.ws.pool = _lib.ptr(self.pool)
        self.args.num_atoms_total, self.args.num_crystals = N, G
        a, p = self.args, _lib.ptr
        a.z_len, a.z_frac, a.u_type = p(self.z_len), p(self.z_frac), p(self.u_type)

    # ------------------------------------------------------------------ buffers
    def _alloc_edges(self, capacity: int) -> None:
        dev, Nc = self.device, self.N_cap
        capacity = max(int(capacity), 1)
        self.edge_capacity = self._edge_alloc = capacity
        self.kernels = self._kernels_flat = None            # release the old slab first: at C3 uncapped one slab is ~100 GB
        self.src = torch.zeros(capacity, dtype=torch.int32, device=dev)
        self.dst = torch.zeros(capacity, dtype=torch.int32, device=dev)
        self.cell = torch.zeros(capacity, dtype=torch.int8, device=dev)
        self.dist = torch.zeros(capacity, dtype=torch.float64, device=dev)
        self.dir = torch.zeros(capacity, 3, dtype=torch.float64, device=dev)
        kdt = torch.float16 if self.precision == "fp16" else torch.float32
        self._kernels_flat = torch.empty(LAYERS * capacity * NUM_ORI * HIDDEN, dtype=kdt, device=dev)
        self.kernels = self._kernels_flat.view(LAYERS, capacity, NUM_ORI, HIDDEN)
        if self.debug and self._debug_flat is None:
            node = Nc * NUM_ORI * HIDDEN
            self._debug_flat = [torch.zeros(LAYERS * node, dtype=torch.float32, device=dev),
                                torch.zeros(LAYERS * node, dtype=torch.float32, device=dev),
                                torch.zeros((LAYERS + 1) * node, dtype=torch.float32, device=dev)]
        if not self.debug:
            self.x1_debug = self.x2_debug = self.h_debug = None
        B = lambda name: self._bufs[name][1]  # noqa: E731
        ws = _lib.Workspace()
        ws.h, ws.y, ws.kernels, ws.acc = B("h").data_ptr(), self.y.data_ptr(), self.kernels.data_ptr(), B("acc").data_ptr()
        ws.x1 = B("x1").data_ptr()
        if self.debug:      # the kernels index these by the CURRENT N (layer stride N * O * C): flat buffers
            ws.x1_debug, ws.x2_debug, ws.h_debug = (t.data_ptr() for t in self._debug_flat)
        else:
            ws.x1_debug = ws.x2_debug = ws.h_debug = None
        ws.edge_capacity = capacity
        ws.onehot_types = None          # set by predict_scores / step: x[:, :Z] is one_hot(self.types) there
        ws.pool = _lib.ptr(self._pool_flat)
        self.ws = ws
        a = _lib.StepArgs()
        p = lambda name: B(name).data_ptr()  # noqa: E731
        a.frac, a.types, a.lengths, a.angles, a.lattice = p("frac"), p("types"), p("lengths"), p("angles"), p("lattice")
        a.angle_trig = p("angle_trig")
        a.atom_offset, a.crystal_of_atom = p("atom_offset"), p("crystal_of_atom")
        a.num_atoms_total, a.num_crystals = self.N, self.G
        a.pos, a.raw_count, a.deg, a.row_ptr = p("pos"), p("raw_count"), p("deg"), p("row_ptr")
        a.num_neighbors_image = p("num_neighbors_image")
        a.src, a.dst, a.cell, a.dist, a.dir = (t.data_ptr() for t in (self.src, self.dst, self.cell, self.dist, self.dir))
        a.overflow_flag = self.overflow_flag.data_ptr()
        a.x, a.vec, a.logits, a.score, a.len0 = p("x"), p("vec"), p("logits"), p("score"), p("len0")
        a.z_len, a.z_frac, a.u_type = p("z_len"), p("z_frac"), p("u_type")
        a.vp_betas, a.fourier_w, a.ve_sigmas = (t.data_ptr() for t in (self.d_vp_betas, self.d_fourier_w, self.d_ve_sigmas))
        a.q_keep, a.q_to_mask = self.d_q_keep.data_ptr(), self.d_q_to_mask.data_ptr()
        a.onestep_keep, a.onestep_to_mask = self.tabs.onestep_keep, self.tabs.onestep_to_mask
        a.emb, a.num_steps, a.cap, a.radius = self.emb, self.tabs.T, self.cap, self.radius
        a.precision, a.update_types = PRECISIONS[self.precision], 1
        self.args = a
        if self.N:                      # re-allocation of a bound engine (uncapped graphs): keep the topology's views
            self.ws.pool = _lib.ptr(self.pool)

    def _bind_edges(self, capacity: int) -> None:
        """Edge capacity the kernels see (<= the allocation): slab layer stride, fill bound, backward row extent."""
        capacity = max(int(capacity), 1)
        assert capacity <= self._edge_alloc
        self.edge_capacity = capacity
        self.kernels = self._kernels_flat[: LAYERS * capacity * NUM_ORI * HIDDEN].view(LAYERS, capacity, NUM_ORI, HIDDEN)
        self.ws.edge_capacity = capacity

    @property
    def stream(self) -> int:
        return torch.cuda.current_stream(self.device).cuda_stream

    # ------------------------------------------------------------------ state
    def set_state(self, frac, types, lengths, angles) -> None:
        """Copies the diffusion state (any float dtype / host or device) into the engine's fp64 buffers."""
        self.frac.copy_(torch.as_tensor(frac).reshape(self.N, 3), non_blocking=True)
        self.types.copy_(torch.as_tensor(types).reshape(self.N), non_blocking=True)
        self.lengths.copy_(torch.as_tensor(lengths).reshape(self.G, 3), non_blocking=True)
        ang = torch.as_tensor(angles).reshape(self.G, 3)
        self.angles.copy_(ang, non_blocking=True)
        self.angle_trig.copy_(angle_factors(ang.detach().to("cpu", torch.float64)), non_blocking=True)

    def set_noise(self, z_len, z_frac, u_type) -> None:
        self.z_len.copy_(torch.as_tensor(z_len).reshape(self.G, 3), non_blocking=True)
        self.z_frac.copy_(torch.as_tensor(z_frac).reshape(self.N, 3), non_blocking=True)
        self.u_type.copy_(torch.as_tensor(u_type).reshape(self.N, self.Z), non_blocking=True)

    def stage_noise(self, z_len, z_frac, u_type) -> None:
        """Upload the NEXT step's noise (pinned host tensors) into the second set of device buffers on a side
        stream, so that the host->device copy (30 MB of uniforms per step at C2) runs under the current step's
        kernels.  `use_staged_noise()` makes the staged set current once the copy has landed;
        `release_noise()` after a step marks the set that step read as reusable."""
        if not hasattr(self, "_noise_sets"):
            other = (torch.empty_like(self.z_len), torch.empty_like(self.z_frac), torch.empty_like(self.u_type))
            self._noise_sets = [(self.z_len, self.z_frac, self.u_type), other]
            self._noise_front = 0
            self._copy_stream = torch.cuda.Stream(self.device)
            self._noise_ready = torch.cuda.Event()
            self._noise_consumed = [torch.cuda.Event(), torch.cuda.Event()]
            for ev in self._noise_consumed:
                ev.record(torch.cuda.current_stream(self.device))
        back = 1 - self._noise_front
        self._copy_stream.wait_event(self._noise_consumed[back])     # the step that read this set has finished
        with torch.cuda.stream(self._copy_stream):
            for dst_, src_, shape in zip(self._noise_sets[back], (z_len, z_frac, u_type),
                                         ((self.G, 3), (self.N, 3), (self.N, self.Z))):
                dst_.copy_(torch.as_tensor(src_).reshape(shape), non_blocking=True)
            self._noise_ready.record(self._copy_stream)

    def use_staged_noise(self) -> None:
        """Swap the staged noise in (device-side wait on the copy; no host synchronisation)."""
        torch.cuda.current_stream(self.device).wait_event(self._noise_ready)
        self._noise_front = 1 - self._noise_front
        self.z_len, self.z_frac, self.u_type = self._noise_sets[self._noise_front]
        a = self.args
        a.z_len, a.z_frac, a.u_type = _lib.ptr(self.z_len), _lib.ptr(self.z_frac), _lib.ptr(self.u_type)

    def release_noise(self) -> None:
        """After enqueueing a step: the noise set it reads may be refilled once the stream gets here."""
        if hasattr(self, "_noise_sets"):
            self._noise_consumed[self._noise_front].record(torch.cuda.current_stream(self.device))

    def draw_noise(self, seed: int, step: int) -> None:
        """Philox noise on the device for throughput runs (the reference draws torch CPU noise)."""
        _lib.call("arreau_step_noise", C.c_uint64(seed), step, self.G, self.N, self.Z, self.z_len.data_ptr(),
                  self.z_frac.data_ptr(), self.u_type.data_ptr(), self.stream)

    # ------------------------------------------------------------------ per-crystal keyed sampling noise
    def set_crystal_ids(self, crystal_ids) -> None:
        """Bind the ids of the bound batch's crystals (G, any integer dtype, host or device): the key of the
        keyed draws below.  Kept on the device next to the topology."""
        ids = torch.as_tensor(crystal_ids).reshape(-1)
        if ids.shape[0] != self.G:
            raise ValueError(f"{ids.shape[0]} crystal ids for a batch of {self.G} crystals")
        ids = ids.to(torch.int64)
        self.crystal_id.copy_(ids.pin_memory() if ids.device.type == "cpu" and self.device.type == "cuda" else ids,
                              non_blocking=True)

    def init_state_keyed(self, seed: int, types, pos_sigma_max: float) -> None:
        """The sampler's initial state drawn per crystal on the device (arreau_sample_init_keyed, keyed by seed and the
        bound crystal ids): angles (90, U(90,180), 90), lengths N(0,1), frac N(0,1) * pos_sigma_max; types are given.
        The angle factors are formed on the host from the drawn angles, as set_state does (one device->host read of
        G x 3 doubles)."""
        _lib.call("arreau_sample_init_keyed", C.c_uint64(int(seed)), self.G, self.N, self.crystal_id.data_ptr(),
                  self.atom_offset.data_ptr(), self.crystal_of_atom.data_ptr(), float(pos_sigma_max),
                  self.angles.data_ptr(), self.lengths.data_ptr(), self.frac.data_ptr(), self.stream)
        self.types.copy_(torch.as_tensor(types).reshape(self.N), non_blocking=True)
        self.angle_trig.copy_(angle_factors(self.angles.to("cpu", torch.float64)), non_blocking=True)

    def draw_noise_keyed(self, seed: int, step: int) -> None:
        """One step's noise drawn per crystal on the device (arreau_sample_noise_keyed, step ordinal `step`)."""
        _lib.call("arreau_sample_noise_keyed", C.c_uint64(int(seed)), int(step), self.G, self.N, self.Z,
                  self.crystal_id.data_ptr(), self.atom_offset.data_ptr(), self.crystal_of_atom.data_ptr(),
                  self.z_len.data_ptr(), self.z_frac.data_ptr(), self.u_type.data_ptr(), self.stream)

    # ------------------------------------------------------------------ graph
    def _count(self) -> None:
        s = self.stream
        _lib.call("arreau_graph_count", self.pos.data_ptr(), self.lattice.data_ptr(), self.atom_offset.data_ptr(),
                  self.crystal_of_atom.data_ptr(), self.N, self.G, self.radius * self.radius, self.cap, 1,
                  self.raw_count.data_ptr(), self.deg.data_ptr(), self.num_neighbors_image.data_ptr(), s)
        _lib.call("arreau_graph_scan", self.deg.data_ptr(), self.row_ptr.data_ptr(), self.N, s)

    def _ensure_capacity(self) -> None:
        """Uncapped graphs only: the edge count is data dependent, so size the buffers from the count
        (one host synchronisation; with a positive cap E <= N*cap and nothing is read back)."""
        if self.cap > 0:
            return
        self._count()
        E = int(self.row_ptr[self.N].item())
        if E > self.edge_capacity:
            self._alloc_edges(int(E * 1.1) + 1024)

    def build_graph(self, edge_index_i64: Optional[torch.Tensor] = None, cell_offsets: Optional[torch.Tensor] = None):
        """lattice/pos must be current.  count -> scan -> fill."""
        s = self.stream
        self._count()
        self.overflow_flag.zero_()
        _lib.call("arreau_graph_fill", self.pos.data_ptr(), self.lattice.data_ptr(), self.atom_offset.data_ptr(),
                  self.crystal_of_atom.data_ptr(), self.N, self.G, self.radius * self.radius, self.cap, 1,
                  self.raw_count.data_ptr(), self.row_ptr.data_ptr(), self.edge_capacity, self.src.data_ptr(),
                  self.dst.data_ptr(), self.cell.data_ptr(), self.dist.data_ptr(), self.dir.data_ptr(),
                  _lib.ptr(edge_index_i64), _lib.ptr(cell_offsets), self.overflow_flag.data_ptr(), s)

    def num_edges(self) -> int:
        return int(self.row_ptr[self.N].item())

    # ------------------------------------------------------------------ predict_scores
    def prepare_inputs(self, t, from_trig: bool = True) -> None:
        """lattice_from_params, feature assembly, frac -> cart (diffusion_loss.py:124-158).  from_trig=False
        evaluates the angle factors on the device (training batches, whose angles come from matrix_to_params)."""
        s = self.stream
        if isinstance(t, int):
            t_ptr, t_scalar = None, t
        else:
            self.t_of_atom.copy_(torch.as_tensor(t).reshape(self.N).to(torch.int32), non_blocking=True)
            t_ptr, t_scalar = self.t_of_atom.data_ptr(), 0
        if from_trig:
            _lib.call("arreau_lattice_from_trig", self.lengths.data_ptr(), self.angle_trig.data_ptr(), self.G,
                      self.lattice.data_ptr(), s)
        else:
            _lib.call("arreau_lattice_from_params", self.lengths.data_ptr(), self.angles.data_ptr(), self.G,
                      self.lattice.data_ptr(), s)
        _lib.call("arreau_assemble_features", self.frac.data_ptr(), self.types.data_ptr(), self.lengths.data_ptr(),
                  self.angles.data_ptr(), self.lattice.data_ptr(), self.atom_offset.data_ptr(),
                  self.crystal_of_atom.data_ptr(), t_ptr, t_scalar, self.d_vp_betas.data_ptr(),
                  self.d_fourier_w.data_ptr(), self.emb, self.N, self.G, self.Z, self.x.data_ptr(),
                  self.vec.data_ptr(), s)
        _lib.call("arreau_frac_to_cart", self.frac.data_ptr(), self.lattice.data_ptr(), self.crystal_of_atom.data_ptr(),
                  self.N, self.pos.data_ptr(), s)

    def forward(self, x=None, vec=None) -> Tuple[torch.Tensor, torch.Tensor, torch.Tensor]:
        """PonitaFiberBundle.forward on the engine's current graph; returns (logits, score, len0) f32."""
        x = self.x if x is None else x
        vec = self.vec if vec is None else vec
        _lib.call("arreau_ponita_forward", self.w.ref(), C.byref(self.ws), PRECISIONS[self.precision], x.data_ptr(),
                  vec.data_ptr(), self.row_ptr.data_ptr(), self.src.data_ptr(), self.dist.data_ptr(),
                  self.dir.data_ptr(), self.lattice.data_ptr(), self.atom_offset.data_ptr(),
                  self.crystal_of_atom.data_ptr(), self.N, self.G, self.radius, self.logits.data_ptr(),
                  self.score.data_ptr(), self.len0.data_ptr(), self.stream)
        return self.logits, self.score, self.len0

    def predict_scores(self, t) -> Tuple[torch.Tensor, torch.Tensor, torch.Tensor]:
        """DiffusionLoss.predict_scores (diffusion_loss.py:112-197) on the engine state.
        Returns (score[N,3], logits[N,Z], len0[G,3]) as fp32 device tensors (views of engine buffers)."""
        self.prepare_inputs(t)
        self._ensure_capacity()
        self.build_graph()
        self.ws.onehot_types = self.types.data_ptr()      # x was assembled from self.types
        try:
            self.forward()
        finally:
            self.ws.onehot_types = None
        return self.score, self.logits, self.len0

    # ------------------------------------------------------------------ step
    def step(self, t: int, update_types: bool = True) -> None:
        """One iteration of the sampler loop (diffusion_loss.py:319-349), in place, using the noise
        currently in z_len / z_frac / u_type.  A single C call, no host synchronisation when cap > 0."""
        tb = self.tabs
        if not (1 <= t <= tb.T):
            raise ValueError(f"timestep {t} outside 1..{tb.T}")
        if self.cap <= 0:
            self.prepare_inputs(t)
            self._ensure_capacity()
        a = self.args
        a.t = int(t)
        a.vp_cx0, a.vp_cxt = float(tb.vp_cx0[t]), float(tb.vp_cxt[t])
        a.vp_denom, a.vp_var = float(tb.vp_denom[t]), float(tb.vp_var[t])
        a.update_types = 1 if update_types else 0
        self.ws.onehot_types = self.types.data_ptr()      # the step assembles x from the state's types
        try:
            _lib.call("arreau_denoise_step", self.w.ref(), C.byref(self.ws), C.byref(a), self.stream)
        finally:
            self.ws.onehot_types = None

    # ------------------------------------------------------------------ whole trajectory as one replayed CUDA graph
    def capture_trajectory_graph(self, t_first: int, seed: int, update_types: bool = True,
                                 keyed: bool = False) -> "torch.cuda.CUDAGraph":
        """Capture ONE denoise step (arreau_denoise_step_replay: Philox noise + graph + network + update, every
        per-step scalar in device memory) as a CUDA graph; replay k runs timestep max(t_first - k, 1) with the noise of
        step ordinal k, so `for _ in range(steps): g.replay()` is the sampler loop of diffusion_loss.py:318-349 with one
        launch per step instead of 26.  Bit-identical to `draw_noise(seed, k); step(t)`, or with `keyed` (the noise
        keyed per crystal by the bound crystal ids) to `draw_noise_keyed(seed, k); step(t)`.  Capped graphs only.
        `reset_trajectory_graph()` rewinds the device-side step counter (a new trajectory on new state)."""
        if self.cap <= 0:
            raise ValueError("the replayable step needs max_neighbors > 0 (uncapped graphs size their buffers on the host)")
        tb, dev = self.tabs, self.device
        if not hasattr(self, "_replay"):
            table = torch.stack([tb.vp_cx0, tb.vp_cxt, tb.vp_denom, tb.vp_var], dim=1).to(torch.float64).contiguous().to(dev)
            self._replay_bufs = dict(counter=torch.zeros(1, dtype=torch.int32, device=dev), table=table,
                                     t_of_atom=torch.zeros(self.N_cap, dtype=torch.int32, device=dev),
                                     dyn=torch.zeros(5, dtype=torch.float64, device=dev),
                                     step_out=torch.zeros(1, dtype=torch.int32, device=dev))
            self._replay = _lib.StepReplay()
        b, r = self._replay_bufs, self._replay
        r.counter, r.vp_table, r.t_of_atom = b["counter"].data_ptr(), b["table"].data_ptr(), b["t_of_atom"].data_ptr()
        r.dyn, r.step_out, r.seed, r.t_first = b["dyn"].data_ptr(), b["step_out"].data_ptr(), int(seed), int(t_first)
        r.crystal_id = self.crystal_id.data_ptr() if keyed else None
        a = self.args
        a.update_types = 1 if update_types else 0
        self.ws.onehot_types = self.types.data_ptr()
        keep = [t.clone() for t in (self.frac, self.types, self.lengths, self.lattice)]

        def one_step():
            _lib.call("arreau_denoise_step_replay", self.w.ref(), C.byref(self.ws), C.byref(a), C.byref(r), self.stream)

        # warm up outside the capture (first launches set function attributes), on a side stream as torch requires
        side = torch.cuda.Stream(dev)
        side.wait_stream(torch.cuda.current_stream(dev))
        with torch.cuda.stream(side):
            one_step()
        torch.cuda.current_stream(dev).wait_stream(side)
        torch.cuda.synchronize(dev)
        g = torch.cuda.CUDAGraph()
        with torch.cuda.graph(g):
            one_step()
        # the warm-up step advanced the state and the counter: restore both
        for dst, src in zip((self.frac, self.types, self.lengths, self.lattice), keep):
            dst.copy_(src)
        b["counter"].zero_()
        self._trajectory_graph = g
        return g

    def reset_trajectory_graph(self) -> None:
        self._replay_bufs["counter"].zero_()

    def kernels_logical(self, layer: int, num_edges: Optional[int] = None) -> torch.Tensor:
        """Spatial kernels of one layer as fp32 [E,O,C] in logical channel order (debug / tests).  The fp16 path
        stores the 16-byte chunk k of row (e, o) at chunk position k ^ o (csrc/model_tc.cu); undo that here."""
        E = self.num_edges() if num_edges is None else num_edges
        k = self.kernels[layer, :E]
        if self.precision != "fp16":
            return k.float()
        k = k.float().view(E, NUM_ORI, HIDDEN // 8, 8)
        o = torch.arange(NUM_ORI, device=k.device)[:, None]
        pos = torch.arange(HIDDEN // 8, device=k.device)[None, :] ^ o          # logical chunk c lives at c ^ o
        return torch.gather(k, 2, pos[None, :, :, None].expand(E, -1, -1, 8)).reshape(E, NUM_ORI, HIDDEN)

    def edges(self):
        """Current edge list as (src, dst, cell, dist, dir) trimmed to E (host synchronisation)."""
        E = self.num_edges()
        if int(self.overflow_flag.item()):
            raise RuntimeError("edge capacity overflow")
        return self.src[:E], self.dst[:E], self.cell[:E], self.dist[:E], self.dir[:E]

    # ------------------------------------------------------------------ measurement
    def timed_breakdown(self, t: int, iters: int = 3):
        """Per-kernel device times (ms, averaged over `iters`) of one predict_scores + update, launched one
        entry point at a time with CUDA events on the current stream.  Leaves the state untouched (the update
        kernels write to scratch).  Used by bench.py for the roofline of the dominant kernel."""
        w, s, Z = self.w.t, None, self.Z
        fp16 = self.precision == "fp16"
        names, fns = [], []

        def add(name, fn):
            names.append(name)
            fns.append(fn)

        add("features", lambda: self.prepare_inputs(t))
        add("graph", lambda: self.build_graph())
        pooled = self.pool is not None
        if pooled:
            add("node_embed", lambda: _lib.call("arreau_node_embed_pooled", self.x.data_ptr(), self.types.data_ptr(), Z,
                                                self.vec.data_ptr(), w["w_embed_t"].data_ptr(), w["ori"].data_ptr(),
                                                self.N, self.F, 4, self.h.data_ptr(), self.pool[0].data_ptr(),
                                                w["readout_v"][0].data_ptr(), self.stream))
        else:
            add("node_embed", lambda: _lib.call("arreau_node_embed_typed", self.x.data_ptr(), self.types.data_ptr(), Z,
                                                self.vec.data_ptr(), w["w_embed_t"].data_ptr(), w["ori"].data_ptr(),
                                                self.N, self.F, 4, self.h.data_ptr(), self.stream))
        nep = self.row_ptr.data_ptr() + 4 * self.N
        if fp16:
            add("edge_kernels", lambda: _lib.call(
                "arreau_edge_kernels_f16", self.dir.data_ptr(), self.dist.data_ptr(), self.lattice.data_ptr(),
                self.crystal_of_atom.data_ptr(), self.src.data_ptr(), nep, self.edge_capacity, w["ori"].data_ptr(),
                w["edge_w1_img"].data_ptr(), w["edge_w_img"].data_ptr(), w["b2"].data_ptr(),
                self.radius, self.kernels.data_ptr(), self.stream))
        else:
            add("edge_kernels", lambda: _lib.call(
                "arreau_edge_kernels_f32", self.dir.data_ptr(), self.dist.data_ptr(), self.lattice.data_ptr(),
                self.crystal_of_atom.data_ptr(), self.src.data_ptr(), nep, self.edge_capacity, w["ori"].data_ptr(),
                w["w1m_t"].data_ptr(), w["w2_t"].data_ptr(), w["b2"].data_ptr(), w["wk_t"].data_ptr(),
                self.radius, self.kernels.data_ptr(), self.stream))
        for l in range(LAYERS):
            if fp16 and self.edge_capacity > 16 * self.N:
                # long rows (uncapped graphs): the step runs the CTA-per-atom gather + tensor-core fiber conv pair
                # (csrc/step.cu); both launches are booked under the fused kernel's label
                add("message_fiber_norm", lambda l=l: _lib.call(
                    "arreau_message_gather", self.kernels[l].data_ptr(), 1, self.h.data_ptr(),
                    self.row_ptr.data_ptr(), self.src.data_ptr(), self.N, 1, self.x1.data_ptr(), self.stream))
                add("message_fiber_norm", lambda l=l: _lib.call(
                    "arreau_fiber_norm", self.x1.data_ptr(), 1, w["fiber_kernel"][l].data_ptr(),
                    w["fiber_frag"].data_ptr() + l * HIDDEN * 32 * 16, w["conv_bias"][l].data_ptr(),
                    w["ln_w"][l].data_ptr(), w["ln_b"][l].data_ptr(), self.N, self.y.data_ptr(), 1, None, self.stream))
            elif fp16:    # one fused launch (the message sums stay in shared memory)
                add("message_fiber_norm", lambda l=l: _lib.call(
                    "arreau_message_fiber_norm_fused", self.kernels[l].data_ptr(), self.h.data_ptr(),
                    self.row_ptr.data_ptr(), self.src.data_ptr(), w["fiber_frag"].data_ptr() + l * HIDDEN * 32 * 16,
                    w["conv_bias"][l].data_ptr(), w["ln_w"][l].data_ptr(), w["ln_b"][l].data_ptr(), self.N,
                    self.y.data_ptr(), None, self.stream))
            else:
                add("message_gather", lambda l=l: _lib.call(
                    "arreau_message_gather", self.kernels[l].data_ptr(), 0, self.h.data_ptr(),
                    self.row_ptr.data_ptr(), self.src.data_ptr(), self.N, 0, self.x1.data_ptr(), self.stream))
                add("fiber_norm", lambda l=l: _lib.call(
                    "arreau_fiber_norm", self.x1.data_ptr(), 0, w["fiber_kernel"][l].data_ptr(), None,
                    w["conv_bias"][l].data_ptr(), w["ln_w"][l].data_ptr(), w["ln_b"][l].data_ptr(), self.N,
                    self.y.data_ptr(), 0, None, self.stream))
            if pooled:
                add("convnext_mlp", lambda l=l: _lib.call(
                    "arreau_convnext_mlp_f16_pooled", self.y.data_ptr(), w["mlp_w_img"].data_ptr() + l * 8 * 32768,
                    w["mlp_b1"][l].data_ptr(), w["mlp_b2"][l].data_ptr(),
                    w["layer_scale"][l].data_ptr(), self.N * NUM_ORI, self.h.data_ptr(), w["ori"].data_ptr(),
                    self.pool[l + 1].data_ptr(), w["readout_v"][l + 1].data_ptr(), Z, self.stream))
            elif fp16:
                add("convnext_mlp", lambda l=l: _lib.call(
                    "arreau_convnext_mlp_f16", self.y.data_ptr(), w["mlp_w_img"].data_ptr() + l * 8 * 32768,
                    w["mlp_b1"][l].data_ptr(), w["mlp_b2"][l].data_ptr(),
                    w["layer_scale"][l].data_ptr(), self.N * NUM_ORI, self.h.data_ptr(), self.stream))
            else:
                add("convnext_mlp", lambda l=l: _lib.call(
                    "arreau_convnext_mlp_f32", self.y.data_ptr(), w["mlp_w1_t"][l].data_ptr(),
                    w["mlp_b1"][l].data_ptr(), w["mlp_w2_t"][l].data_ptr(), w["mlp_b2"][l].data_ptr(),
                    w["layer_scale"][l].data_ptr(), self.N * NUM_ORI, self.h.data_ptr(), self.stream))
            if not pooled:
                add("readout", lambda l=l: _lib.call(
                    "arreau_readout_accumulate", self.h.data_ptr(), w["wr_t"][l].data_ptr(), w["br"][l].data_ptr(),
                    w["ori"].data_ptr(), self.N, Z, int(l == 0), self.acc.data_ptr(), self.stream))
        if pooled:
            add("readout", lambda: _lib.call("arreau_readout_pooled", self.pool.data_ptr(), w["readout_v"].data_ptr(),
                                             w["readout_bias"].data_ptr(), self.N, Z, LAYERS + 1,
                                             self.acc.data_ptr(), self.stream))
        add("readout", lambda: _lib.call("arreau_readout_finalize", self.acc.data_ptr(), self.atom_offset.data_ptr(),
                                         self.N, self.G, Z, 1 if pooled else LAYERS, self.logits.data_ptr(), self.score.data_ptr(),
                                         self.len0.data_ptr(), self.stream))
        sc_len, sc_frac, sc_types = torch.empty_like(self.lengths), torch.empty_like(self.frac), torch.empty_like(self.types)
        tb = self.tabs

        def update():
            _lib.call("arreau_vp_lattice_reverse", self.lengths.data_ptr(), self.len0.data_ptr(),
                      self.atom_offset.data_ptr(), self.z_len.data_ptr(), t, float(tb.vp_cx0[t]), float(tb.vp_cxt[t]),
                      float(tb.vp_denom[t]), float(tb.vp_var[t]), self.G, sc_len.data_ptr(), self.stream)
            _lib.call("arreau_ve_pbc_reverse", self.frac.data_ptr(), self.score.data_ptr(), self.z_frac.data_ptr(),
                      None, t, self.d_ve_sigmas.data_ptr(), self.N, sc_frac.data_ptr(), self.stream)
            _lib.call("arreau_d3pm_reverse", self.types.data_ptr(), self.logits.data_ptr(), self.u_type.data_ptr(), None,
                      t, self.d_q_keep.data_ptr(), self.d_q_to_mask.data_ptr(), tb.onestep_keep, tb.onestep_to_mask,
                      tb.T, self.N, Z, sc_types.data_ptr(), self.stream)
        add("update", update)
        totals, counts = {}, {}
        for it in range(iters + 1):          # first pass is warm-up
            evs = []
            for fn in fns:
                a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                a.record()
                fn()
                b.record()
                evs.append((a, b))
            torch.cuda.synchronize(self.device)
            if it == 0:
                continue
            for name, (a, b) in zip(names, evs):
                totals[name] = totals.get(name, 0.0) + a.elapsed_time(b)
                counts[name] = counts.get(name, 0) + 1
        launches = {n: counts[n] // iters for n in counts}
        return {n: dict(ms_per_step=totals[n] / iters, launches_per_step=launches[n],
                        ms_per_launch=totals[n] / counts[n]) for n in totals}
