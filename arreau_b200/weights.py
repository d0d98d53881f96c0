"""Reference state_dict -> device weight layouts of the kernels.

Parameter names are the reference's (SURVEY 8b): basis_fn.{1,3}.*, fiber_basis_fn.{1,3}.*, x_embedder.weight,
interaction_layers.{l}.{layer_scale, conv.bias, conv.kernel.weight, conv.fiber_kernel.weight, linear_1.*,
linear_2.*, norm.*}, read_out_layers.{l}.*.  The orientation grid is not part of the state_dict (quirk B2)
and is passed explicitly.
"""
from __future__ import annotations

import ctypes as C
import math
from typing import Dict, Mapping

import numpy as np
import torch

from . import _lib

NUM_ORI, HIDDEN, BASIS, WIDEN, LAYERS = 16, 128, 256, 4, 5
NUM_MONO, MONO_PAD = 83, 96


def monomial_fold_table(num_in: int = 6, degree: int = 3) -> np.ndarray:
    """Index of the distinct monomial each PolynomialFeatures(3) output equals
    (ponita/nn/embedding.py:10-14: [x, x(x)x, (x(x)x)(x)x], index = previous*6 + j).
    Monomial order = csrc/common.cuh monomials83(): all i, all i<=j, all i<=j<=k."""
    assert num_in == 6 and degree == 3
    ids: Dict[tuple, int] = {}
    for i in range(6):
        ids[(i,)] = len(ids)
    for i in range(6):
        for j in range(i, 6):
            ids[(i, j)] = len(ids)
    for i in range(6):
        for j in range(i, 6):
            for k in range(j, 6):
                ids[(i, j, k)] = len(ids)
    assert len(ids) == NUM_MONO
    table = []
    for i in range(6):
        table.append(ids[(i,)])
    for i in range(6):
        for j in range(6):
            table.append(ids[tuple(sorted((i, j)))])
    for i in range(6):
        for j in range(6):
            for k in range(6):
                table.append(ids[tuple(sorted((i, j, k)))])
    return np.asarray(table, dtype=np.int64)   # [258]


def umma_tile_image(w: np.ndarray) -> torch.Tensor:
    """[rows, K] fp weights (rows = the UMMA N index, K a multiple of 64) -> the fp16 shared-memory image the
    tcgen05 kernels expect (csrc/tc_common.cuh): K slabs of 64 back to back, each `rows` rows of 128 bytes with
    the 16-byte chunk c of row r stored at chunk position c ^ (r & 7).  Returned as a flat int16 CPU tensor."""
    rows, K = w.shape
    assert K % 64 == 0 and rows % 8 == 0
    bits = torch.as_tensor(np.ascontiguousarray(w), dtype=torch.float32).to(torch.float16).view(torch.int16).numpy()
    t = bits.reshape(rows, K // 64, 8, 8).transpose(1, 0, 2, 3)          # [slab, row, chunk, 8]
    pos = np.arange(8)[None, :] ^ (np.arange(rows)[:, None] & 7)          # out[.., r, p] = in[.., r, p ^ (r & 7)]
    out = np.take_along_axis(t, pos[None, :, :, None], axis=2)
    return torch.as_tensor(np.ascontiguousarray(out).reshape(-1))


def _np(v) -> np.ndarray:
    if isinstance(v, torch.Tensor):
        return v.detach().cpu().double().numpy()
    return np.asarray(v, dtype=np.float64)


def pooled_readout_weights(wr: np.ndarray, br: np.ndarray, ori: np.ndarray):
    """Combined matrices of the pooled read-out (arreau_readout_pooled).  wr[L,R,C], br[L,R] with R = Z + 4 rows
    (Z scalars | 1 vector channel | 3 global scalars, ponita.py:111); ori[O,3].  The feature after layer l is
    pool[0] + ... + pool[l] (embedding + residual updates), and the result is the mean over layers of the read-outs
    (ponita.py:108), so entry k meets V_k = (1/L) sum_{l >= max(k,1)} Wr_l.  Columns follow acc[N][Z+6]:
    Z logits | 3 score components (all three use weight row Z, applied to the vector-pooled parts) | 3 length channels.
    The vector channel's bias meets mean_o ori_o (to_from_sphere.py:10-11)."""
    L, R, Cc = wr.shape
    Z = R - 4
    rows = np.concatenate([np.arange(Z), [Z, Z, Z], np.arange(Z + 1, Z + 4)])
    v = np.zeros((L + 1, Cc, Z + 6))
    for k in range(L + 1):
        v[k] = wr[max(k, 1) - 1:].sum(0)[rows].T / L
    bias = br.sum(0)[rows] / L
    bias[Z:Z + 3] *= ori.mean(0)
    return v, bias


class PonitaWeights:
    """Device copies of one PonitaFiberBundle's parameters in kernel layouts."""

    def __init__(self, state: Mapping[str, object], ori_grid, device="cuda", with_f16: bool = True):
        sd = {k: _np(v) for k, v in state.items() if hasattr(v, "shape") and np.prod(np.shape(v)) > 0
              and not k.endswith("callibrated") and not k.startswith("windowing_fn")}
        self.device = torch.device(device)
        ori = _np(ori_grid)
        if ori.shape != (NUM_ORI, 3):
            raise ValueError(f"unsupported orientation grid {ori.shape}: kernels are specialised on {NUM_ORI}")
        w1 = sd["basis_fn.1.weight"]
        if w1.shape != (HIDDEN, 258) or sd["basis_fn.3.weight"].shape != (BASIS, HIDDEN):
            raise ValueError("unsupported model dims: kernels are specialised on hidden 128 / basis 256 / degree 3")
        if sd["fiber_basis_fn.1.weight"].shape != (HIDDEN, 3):
            raise ValueError("unsupported fiber basis input width")
        L = LAYERS
        for l in range(L):
            if f"interaction_layers.{l}.conv.kernel.weight" not in sd:
                raise ValueError(f"expected {L} interaction layers")
        if f"interaction_layers.{L}.conv.kernel.weight" in sd:
            raise ValueError(f"unsupported number of layers (kernels are specialised on {L})")
        fold = monomial_fold_table()
        w1m = np.zeros((HIDDEN, NUM_MONO))
        np.add.at(w1m, (slice(None), fold), w1)           # sum the columns of equal monomials (fp64)
        w1m_t = np.zeros((MONO_PAD, HIDDEN))
        w1m_t[:NUM_MONO] = w1m.T
        w1m_t[NUM_MONO] = sd["basis_fn.1.bias"]            # constant-1 monomial carries the bias
        stack = lambda name: np.stack([sd[name.format(l=l)] for l in range(L)])  # noqa: E731
        lay = lambda name: stack(f"interaction_layers.{{l}}.{name}")  # noqa: E731
        f32 = lambda a: torch.as_tensor(np.ascontiguousarray(a), dtype=torch.float32).to(self.device)  # noqa: E731
        self._fp32_layouts(lambda name: f32(stack(name) if "{l}" in name else sd[name]), f32(w1m_t), f32(ori))
        stream = torch.cuda.current_stream(self.device).cuda_stream
        if with_f16:   # fp16 mma fragments of the fiber kernels for the tensor-core fiber conv
            self.t["fiber_frag"] = torch.empty(L * HIDDEN * 32 * 4, dtype=torch.int32, device=self.device)
            _lib.call("arreau_fiber_frag_pack", self.t["fiber_kernel"].data_ptr(), L, self.t["fiber_frag"].data_ptr(), stream)
        torch.cuda.current_stream(self.device).synchronize()
        if with_f16:
            # tcgen05 path: every weight tile as a ready-to-copy UMMA shared-memory image
            w1pad = np.zeros((HIDDEN, 128))
            w1pad[:, :MONO_PAD] = w1m_t.T                                  # [N = hidden, K = 96 -> 128]
            # the kernels' packed-fp16 GELU returns 2 gelu(x) (csrc/tc_common.cuh gelu2_f16): every matrix that consumes a
            # GELU output carries the factor 1/2 (a power of two: exact in fp16)
            w2 = 0.5 * np.asarray(sd["basis_fn.3.weight"])                 # [D, C]
            chunks = [umma_tile_image(w2[nh * 128:(nh + 1) * 128, ks * 64:(ks + 1) * 64])
                      for nh in range(2) for ks in range(2)]
            wk = lay("conv.kernel.weight")                                 # [L,C,D]
            chunks += [umma_tile_image(0.5 * wk[l][:, ks * 64:(ks + 1) * 64]) for l in range(L) for ks in range(4)]
            m1, m2 = lay("linear_1.weight"), 0.5 * lay("linear_2.weight")  # [L,4C,C], [L,C,4C]
            mlp = []
            for l in range(L):
                g1 = [umma_tile_image(m1[l][j * 128:(j + 1) * 128, :]) for j in range(4)]
                g2 = [umma_tile_image(m2[l][:, j * 128:(j + 1) * 128]) for j in range(4)]
                mlp += [g1[0], g1[1], g2[0], g1[2], g2[1], g1[3], g2[2], g2[3]]   # MMA issue order
            self.t.update(edge_w1_img=umma_tile_image(w1pad).to(self.device),
                          edge_w_img=torch.cat(chunks).to(self.device), mlp_w_img=torch.cat(mlp).to(self.device))
            rv, rb = pooled_readout_weights(stack("read_out_layers.{l}.weight"), stack("read_out_layers.{l}.bias"), ori)
            self.t.update(readout_v=f32(rv), readout_bias=f32(rb))
        self._fill_struct()

    @classmethod
    def from_flat(cls, flat, ori_grid: torch.Tensor) -> "PonitaWeights":
        """Kernel layouts of the fp32 path straight from the training step's flat parameter buffer (training.py
        FlatParams, arreau_train_layout_t order): tensors whose kernel layout equals the reference's own layout are
        VIEWS of the flat buffer (no copy, so they are current after every optimizer step by construction), the six
        transposed matrices are one strided copy each, plus the monomial fold and the fiber-kernel precompute --
        ~10 launches per step."""
        self = cls.__new__(cls)
        dev = flat.data.device
        self.device = dev

        def get(name):
            off, shape = flat.specs[name.format(l=0)]
            if "{l}" in name:      # the flat layout keeps a tensor's layers consecutive: one [L, ...] view
                shape = (LAYERS,) + shape
            return flat.data[off:off + math.prod(shape)].view(*shape)

        fold = getattr(flat, "_fold_table", None)
        if fold is None:
            fold = flat._fold_table = torch.as_tensor(monomial_fold_table(), dtype=torch.int32).to(dev)
        w1m_t = torch.empty(MONO_PAD, HIDDEN, dtype=torch.float32, device=dev)
        _lib.call("arreau_fold_basis_w1", get("basis_fn.1.weight").data_ptr(), get("basis_fn.1.bias").data_ptr(),
                  fold.data_ptr(), w1m_t.data_ptr(), torch.cuda.current_stream(dev).cuda_stream)
        self._fp32_layouts(get, w1m_t, ori_grid.to(dev, torch.float32).contiguous())
        self._fill_struct()
        return self

    def _fp32_layouts(self, get, w1m_t: torch.Tensor, ori: torch.Tensor) -> None:
        """`self.t`: the fp32 kernel layouts, and the fiber kernels evaluated on the device.  get(name) returns a
        parameter under its reference name as an fp32 device tensor; a name with "{l}" stands for that tensor of every
        interaction or read-out layer, stacked [L, ...].  w1m_t: basis_fn.1 folded onto the distinct monomials
        [MONO_PAD, HIDDEN], the bias in row NUM_MONO."""
        L = LAYERS
        lay = lambda name: get(f"interaction_layers.{{l}}.{name}")  # noqa: E731
        wemb, wr = get("x_embedder.weight"), get("read_out_layers.{l}.weight")   # [C, F+V], [L,R,C]
        self.num_readout = wr.shape[1]
        self.num_states = self.num_readout - 4             # scalars | 1 vector | 0 global vec | 3 global scalars
        self.num_vec = 4
        self.num_scalar = wemb.shape[1] - self.num_vec
        self.t: Dict[str, torch.Tensor] = dict(
            ori=ori, w_embed_t=wemb.t().contiguous(), w1m_t=w1m_t, w2_t=get("basis_fn.3.weight").t().contiguous(),
            b2=get("basis_fn.3.bias"),
            wk_t=lay("conv.kernel.weight").permute(2, 0, 1).reshape(BASIS, L * HIDDEN).contiguous(),
            conv_bias=lay("conv.bias"), ln_w=lay("norm.weight"), ln_b=lay("norm.bias"),
            mlp_w1_t=lay("linear_1.weight").transpose(1, 2).contiguous(), mlp_b1=lay("linear_1.bias"),
            mlp_w2_t=lay("linear_2.weight").transpose(1, 2).contiguous(), mlp_b2=lay("linear_2.bias"),
            layer_scale=lay("layer_scale"), wr_t=wr.transpose(1, 2).contiguous(), br=get("read_out_layers.{l}.bias"),
            fiber_kernel=torch.empty(L, NUM_ORI, NUM_ORI, HIDDEN, dtype=torch.float32, device=self.device))
        # K3': input-independent fiber kernels, evaluated once on the device
        fiber = [get("fiber_basis_fn.1.weight"), get("fiber_basis_fn.1.bias"), get("fiber_basis_fn.3.weight"),
                 get("fiber_basis_fn.3.bias"), lay("conv.fiber_kernel.weight")]
        _lib.call("arreau_fiber_kernel_precompute", ori.data_ptr(), *[f.data_ptr() for f in fiber],
                  self.t["fiber_kernel"].data_ptr(), torch.cuda.current_stream(self.device).cuda_stream)

    def _fill_struct(self) -> None:
        self.c = _lib.Weights()
        for name, _ in _lib.Weights._fields_:
            if name in self.t:
                setattr(self.c, name, self.t[name].data_ptr())
        self.c.num_scalar, self.c.num_vec, self.c.num_states = self.num_scalar, self.num_vec, self.num_states

    def ref(self):
        return C.byref(self.c)
