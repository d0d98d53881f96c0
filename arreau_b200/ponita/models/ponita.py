"""Mirror of ponita/models/ponita.py: PonitaFiberBundle with the reference's constructor, parameter names
(so a reference state_dict loads by name) and forward(graph) contract; the forward itself is
arreau_ponita_forward (K2..K7 as sm_100a kernels)."""
from __future__ import annotations

import ctypes as C
import math

import numpy as np
import torch
import torch.nn as nn

from ... import _lib
from ...weights import HIDDEN, LAYERS, NUM_ORI, PonitaWeights


def fibonacci_grid_s2(n: int) -> torch.Tensor:
    """A deterministic quasi-uniform S2 grid.  The reference draws a random grid and relaxes it by 100 SGD steps
    at construction (rotation.py:947-1009) and never checkpoints it (quirk B2); pass the reference's grid via
    `ori_grid=` / `set_orientation_grid` to reproduce a given reference model."""
    i = np.arange(n) + 0.5
    phi = np.arccos(1 - 2 * i / n)
    theta = np.pi * (1 + 5 ** 0.5) * i
    return torch.tensor(np.stack([np.cos(theta) * np.sin(phi), np.sin(theta) * np.sin(phi), np.cos(phi)], 1))


class _Identity(nn.Module):
    pass


class _ConvParams(nn.Module):
    """ponita/nn/conv.py:87-103 parameter container."""

    def __init__(self, hidden, basis):
        super().__init__()
        self.kernel = nn.Linear(basis, hidden, bias=False)
        self.fiber_kernel = nn.Linear(basis, hidden, bias=False)
        self.bias = nn.Parameter(torch.zeros(hidden))
        self.register_buffer("callibrated", torch.tensor(False))   # conv.py:103; set by the callibrate pass


class _ConvNextParams(nn.Module):
    """ponita/nn/convnext.py:7-18 parameter container."""

    def __init__(self, hidden, basis, widening, layer_scale):
        super().__init__()
        self.conv = _ConvParams(hidden, basis)
        self.linear_1 = nn.Linear(hidden, widening * hidden)
        self.linear_2 = nn.Linear(widening * hidden, hidden)
        self.norm = nn.LayerNorm(hidden)
        self.layer_scale = nn.Parameter(torch.ones(hidden) * (layer_scale if layer_scale is not None else 1.0))


class PonitaFiberBundle(nn.Module):
    """ponita/models/ponita.py:29-123."""

    def __init__(self, input_dim, hidden_dim, output_dim, output_dim_global_scalar, output_dim_global_vec,
                 output_dim_edge_scalar, num_layers, output_dim_vec=0, radius=None, num_ori=20, basis_dim=None,
                 degree=3, widening_factor=4, layer_scale=None, task_level="graph", multiple_readouts=True,
                 ori_grid=None, precision="fp32", **kwargs):
        super().__init__()
        basis_dim = hidden_dim if basis_dim is None else basis_dim
        if (hidden_dim, basis_dim, num_ori, num_layers, degree, widening_factor) != (HIDDEN, 256, NUM_ORI, LAYERS, 3, 4):
            raise NotImplementedError("kernels are specialised on hidden 128 / basis 256 / 16 orientations / 5 layers "
                                      "/ degree 3 / widening 4 (main_diffusion.py:88-120)")
        if output_dim_global_vec != 0 or output_dim_edge_scalar != 0 or output_dim_vec != 1 or not multiple_readouts:
            raise NotImplementedError("only the diffusion read-out layout (Z scalars, 1 vector, 3 global scalars) "
                                      "of lightning_wrappers/diffusion.py:69-102 is implemented")
        self.radius, self.num_ori, self.precision = radius, num_ori, precision
        self.output_dim, self.output_dim_vec, self.output_dim_global_scalar = output_dim, output_dim_vec, output_dim_global_scalar
        self.num_layers = num_layers
        in_ch = input_dim[0] + input_dim[1] if isinstance(input_dim, (tuple, list)) else input_dim
        act = nn.GELU()
        self.basis_fn = nn.Sequential(_Identity(), nn.Linear(6 + 36 + 216, hidden_dim), act, nn.Linear(hidden_dim, basis_dim), act)
        self.fiber_basis_fn = nn.Sequential(_Identity(), nn.Linear(3, hidden_dim), act, nn.Linear(hidden_dim, basis_dim), act)
        self.x_embedder = nn.Linear(in_ch, hidden_dim, bias=False)
        self.interaction_layers = nn.ModuleList(
            [_ConvNextParams(hidden_dim, basis_dim, widening_factor, layer_scale) for _ in range(num_layers)])
        n_out = output_dim + output_dim_vec + output_dim_global_vec + output_dim_global_scalar
        self.read_out_layers = nn.ModuleList([nn.Linear(hidden_dim, n_out) for _ in range(num_layers)])
        self.register_buffer("ori_grid", (fibonacci_grid_s2(num_ori) if ori_grid is None else torch.as_tensor(ori_grid)).double(),
                             persistent=False)
        self._packed = None
        self._ws = None
        self.flat = None

    # -- weights ------------------------------------------------------------------------------
    def set_orientation_grid(self, ori_grid) -> None:
        self.ori_grid = torch.as_tensor(ori_grid).double().to(self.ori_grid.device)
        self._packed = None

    def load_state_dict(self, state_dict, strict: bool = True, **kw):
        own = self.state_dict()
        sd = {k: v for k, v in state_dict.items() if k in own and tuple(v.shape) == tuple(own[k].shape)}
        self._packed = None
        return super().load_state_dict(sd, strict=False, **kw)

    def flatten_parameters(self, device, into=None):
        """Re-home every trainable tensor into ONE flat fp32 CUDA buffer (arreau_train_layout_t order, see
        arreau_b200/training.py FlatParams): the nn.Parameters become views of it, keep their reference names, and an
        optimizer / gradient all-reduce sees a single tensor.  into: an existing FlatParams of this layout whose contents
        become the weights (nothing is copied into it).  Returns the FlatParams (also kept as `self.flat`)."""
        from ...training import FlatParams
        n_out = self.read_out_layers[0].out_features
        flat = into if into is not None else FlatParams(self.x_embedder.in_features - 4, 4, n_out - 4, device)
        views = flat.views()
        with torch.no_grad():
            for name, p in self.named_parameters():
                if p.numel() == 0:
                    continue
                if into is None:
                    views[name].copy_(p.detach().to(torch.float32))
                p.data = views[name]
                p.grad = None
        self.flat = flat
        self._packed = None
        return flat

    def pack(self, device) -> PonitaWeights:
        """(Re)build the kernel weight layouts; call after changing parameters in place."""
        self._packed = PonitaWeights(self.state_dict(), self.ori_grid, device=device)
        return self._packed

    # -- forward ------------------------------------------------------------------------------
    @torch.no_grad()
    def forward(self, graph):
        """graph.{x[N,F], vec[N,V,3], edge_index[2,E], dists[E], inter_atom_direction[E,3], lattice[G,3,3],
        batch[N]} (diffusion_loss.py:156-180) -> (scalar[N,Z], vec[N,1,3], global_scalar[G,3], None, [None]*L)."""
        x = graph.x
        if not x.is_cuda:
            raise RuntimeError("arreau_b200 runs on CUDA tensors only (no CPU fallback)")
        dev = x.device
        w = self._packed if self._packed is not None and self._packed.device == dev else self.pack(dev)
        out_dtype = x.dtype
        N = x.shape[0]
        lattice = graph.lattice.to(torch.float64).contiguous()
        G = lattice.shape[0]
        batch = graph.batch.to(dev, torch.int64)
        ei = graph.edge_index.to(dev)
        E = ei.shape[1]
        dst = ei[1]
        if E > 1 and bool((dst[1:] < dst[:-1]).any()):          # reference graphs are already receiver-major
            order = torch.sort(dst, stable=True)[1]
        else:
            order = None
        pick = (lambda t: t) if order is None else (lambda t: t[order])
        src = pick(ei[0]).to(torch.int32).contiguous()
        dist = pick(graph.dists).to(torch.float64).contiguous()
        direction = pick(graph.inter_atom_direction).to(torch.float64).contiguous()
        row_ptr = torch.zeros(N + 1, dtype=torch.int64, device=dev)
        row_ptr[1:] = torch.cumsum(torch.bincount(dst, minlength=N), 0)
        row_ptr = row_ptr.to(torch.int32)
        atom_offset = torch.zeros(G + 1, dtype=torch.int64, device=dev)
        atom_offset[1:] = torch.cumsum(torch.bincount(batch, minlength=G), 0)
        atom_offset = atom_offset.to(torch.int32)
        coa = batch.to(torch.int32).contiguous()
        fp16 = self.precision == "fp16"
        cap = max(E, 1)
        f32 = lambda *s: torch.empty(*s, dtype=torch.float32, device=dev)  # noqa: E731
        ws = _lib.Workspace()
        h, acc, x1 = f32(N, NUM_ORI, HIDDEN), f32(N, w.num_states + 6), f32(N, NUM_ORI, HIDDEN)
        if fp16:     # 128-row UMMA tile images
            y = torch.zeros(((N * NUM_ORI + 127) // 128) * 128 * HIDDEN, dtype=torch.float16, device=dev)
        else:
            y = torch.empty(N, NUM_ORI, HIDDEN, dtype=torch.float32, device=dev)
        kern = torch.empty(LAYERS, cap, NUM_ORI, HIDDEN, dtype=torch.float16 if fp16 else torch.float32, device=dev)
        ws.h, ws.y, ws.kernels, ws.acc, ws.edge_capacity = h.data_ptr(), y.data_ptr(), kern.data_ptr(), acc.data_ptr(), cap
        ws.x1 = x1.data_ptr()
        logits, score, len0 = f32(N, w.num_states), f32(N, 3), f32(G, 3)
        xf = x.to(torch.float32).contiguous()
        vf = graph.vec.to(torch.float32).contiguous()
        _lib.call("arreau_ponita_forward", w.ref(), C.byref(ws), _lib.PRECISION_FP16 if fp16 else _lib.PRECISION_FP32,
                  xf.data_ptr(), vf.data_ptr(), row_ptr.data_ptr(), src.data_ptr(), dist.data_ptr(),
                  direction.data_ptr(), lattice.data_ptr(), atom_offset.data_ptr(), coa.data_ptr(), N, G,
                  float(self.radius), logits.data_ptr(), score.data_ptr(), len0.data_ptr(),
                  torch.cuda.current_stream(dev).cuda_stream)
        return (logits.to(out_dtype), score.to(out_dtype).unsqueeze(1), len0.to(out_dtype), None,
                [None] * self.num_layers)
