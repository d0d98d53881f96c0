"""ctypes binding of libarreau_b200.so -- the only way the Python mirrors reach the GPU.

There is deliberately no fallback: if the library is missing this module raises, and every wrapper
turns a non-zero return code into a RuntimeError (SURVEY 8b: negative = bad arguments, positive =
cudaError_t of a failed launch).
"""
from __future__ import annotations

import ctypes as C
import os

from . import build as _build

_lib = None

c_f32p = C.c_void_p
vp = C.c_void_p
i32 = C.c_int32
i64 = C.c_int64
f64 = C.c_double

ERRORS = {-1: "ARREAU_ERR_BAD_SHAPE", -2: "ARREAU_ERR_UNSUPPORTED", -3: "ARREAU_ERR_WORKSPACE", -4: "ARREAU_ERR_NULL"}
PRECISION_FP32, PRECISION_FP16, PRECISION_TF32 = 0, 1, 2


class Weights(C.Structure):
    _fields_ = [(n, vp) for n in (
        "ori", "w_embed_t", "w1m_t", "w2_t", "b2", "wk_t", "fiber_kernel", "fiber_frag", "conv_bias", "ln_w", "ln_b",
        "mlp_w1_t", "mlp_b1", "mlp_w2_t", "mlp_b2", "layer_scale", "wr_t", "br",
        "edge_w1_img", "edge_w_img", "mlp_w_img", "readout_v", "readout_bias")] + [
        ("num_scalar", i32), ("num_vec", i32), ("num_states", i32), ("reserved", i32)]


class Workspace(C.Structure):
    _fields_ = [("h", vp), ("y", vp), ("kernels", vp), ("acc", vp), ("x1", vp), ("x1_debug", vp), ("x2_debug", vp),
                ("h_debug", vp), ("edge_capacity", i64), ("onehot_types", vp), ("pool", vp)]


class StepArgs(C.Structure):
    _fields_ = [
        ("frac", vp), ("types", vp), ("lengths", vp), ("angles", vp), ("angle_trig", vp), ("lattice", vp),
        ("atom_offset", vp), ("crystal_of_atom", vp), ("num_atoms_total", i32), ("num_crystals", i32),
        ("pos", vp), ("raw_count", vp), ("deg", vp), ("row_ptr", vp), ("num_neighbors_image", vp),
        ("src", vp), ("dst", vp), ("cell", vp), ("dist", vp), ("dir", vp), ("overflow_flag", vp),
        ("x", vp), ("vec", vp), ("logits", vp), ("score", vp), ("len0", vp),
        ("z_len", vp), ("z_frac", vp), ("u_type", vp),
        ("vp_betas", vp), ("fourier_w", vp), ("ve_sigmas", vp), ("q_keep", vp), ("q_to_mask", vp),
        ("onestep_keep", f64), ("onestep_to_mask", f64),
        ("vp_cx0", f64), ("vp_cxt", f64), ("vp_denom", f64), ("vp_var", f64),
        ("emb", i32), ("num_steps", i32), ("t", i32), ("cap", i32), ("radius", f64),
        ("precision", i32), ("update_types", i32), ("allowed_states", vp),
        ("known_atom", vp), ("known_frac", vp), ("known_crystal", vp), ("known_lengths", vp), ("vp_alpha_bars", vp)]


class StepReplay(C.Structure):
    _fields_ = [("counter", vp), ("vp_table", vp), ("t_of_atom", vp), ("dyn", vp), ("step_out", vp),
                ("seed", C.c_uint64), ("t_first", i32), ("reserved", i32), ("crystal_id", vp)]


class WorkspaceSizes(C.Structure):
    FIELDS = ("h", "y", "kernels", "acc", "x1", "debug_per_layer", "pool", "x", "vec", "logits", "score", "len0", "pos",
              "raw_count", "deg", "row_ptr", "num_neighbors_image", "src", "dst", "cell", "dist", "dir", "z_len", "z_frac",
              "u_type")
    _fields_ = [(n, i64) for n in FIELDS]


class TrainLayout(C.Structure):
    FIELDS = ("basis_w1", "basis_b1", "basis_w2", "basis_b2", "fiber_w1", "fiber_b1", "fiber_w2", "fiber_b2", "embed_w",
              "layer_scale", "conv_bias", "conv_kernel_w", "conv_fiber_w", "lin1_w", "lin1_b", "lin2_w", "lin2_b",
              "norm_w", "norm_b", "readout_w", "readout_b", "total")
    _fields_ = [(n, i64) for n in FIELDS]


# name -> argtypes (restype is int unless noted); must list every symbol include/arreau_b200.h declares
SIGNATURES = {
    "arreau_abi_version": [],
    "arreau_model_dims": [C.POINTER(C.c_int)] * 5,
    "arreau_launch_count": [],
    "arreau_workspace_bytes": [i32, i32, i64, i32, i32, i32, C.POINTER(WorkspaceSizes)],
    "arreau_graph_count": [vp, vp, vp, vp, i32, i32, f64, i32, i32, vp, vp, vp, vp],
    "arreau_graph_scan": [vp, vp, i32, vp],
    "arreau_graph_fill": [vp, vp, vp, vp, i32, i32, f64, i32, i32, vp, vp, i64, vp, vp, vp, vp, vp, vp, vp, vp, vp],
    "arreau_lattice_from_params": [vp, vp, i32, vp, vp],
    "arreau_lattice_from_trig": [vp, vp, i32, vp, vp],
    "arreau_frac_to_cart": [vp, vp, vp, i32, vp, vp],
    "arreau_assemble_features": [vp, vp, vp, vp, vp, vp, vp, vp, i32, vp, vp, i32, i32, i32, i32, vp, vp, vp],
    "arreau_fiber_kernel_precompute": [vp] * 8,
    "arreau_node_embed": [vp, vp, vp, vp, i32, i32, i32, vp, vp],
    "arreau_node_embed_typed": [vp, vp, i32, vp, vp, vp, i32, i32, i32, vp, vp],
    "arreau_edge_kernels_f32": [vp, vp, vp, vp, vp, vp, i64, vp, vp, vp, vp, vp, f64, vp, vp],
    "arreau_edge_kernels_f16": [vp, vp, vp, vp, vp, vp, i64, vp, vp, vp, vp, f64, vp, vp],
    "arreau_message_fiber_norm": [vp, i32, vp, vp, vp, vp, vp, vp, vp, vp, i32, vp, i32, vp, vp, vp],
    "arreau_fiber_frag_pack": [vp, i32, vp, vp],
    "arreau_message_fiber_norm_fused": [vp, vp, vp, vp, vp, vp, vp, vp, i32, vp, vp, vp],
    "arreau_message_gather": [vp, i32, vp, vp, vp, i32, i32, vp, vp],
    "arreau_fiber_norm": [vp, i32, vp, vp, vp, vp, vp, i32, vp, i32, vp, vp],
    "arreau_convnext_mlp_f32": [vp, vp, vp, vp, vp, vp, i64, vp, vp],
    "arreau_convnext_mlp_f16": [vp, vp, vp, vp, vp, i64, vp, vp],
    "arreau_readout_accumulate": [vp, vp, vp, vp, i32, i32, i32, vp, vp],
    "arreau_node_embed_pooled": [vp, vp, i32, vp, vp, vp, i32, i32, i32, vp, vp, vp, vp],
    "arreau_convnext_mlp_f16_pooled": [vp, vp, vp, vp, vp, i64, vp, vp, vp, vp, i32, vp],
    "arreau_readout_pooled": [vp, vp, vp, i32, i32, i32, vp, vp],
    "arreau_readout_finalize": [vp, vp, i32, i32, i32, i32, vp, vp, vp, vp],
    "arreau_ponita_forward": [C.POINTER(Weights), C.POINTER(Workspace), i32, vp, vp, vp, vp, vp, vp, vp, vp, vp,
                              i32, i32, f64, vp, vp, vp, vp],
    "arreau_vp_lattice_reverse": [vp, vp, vp, vp, i32, f64, f64, f64, f64, i32, vp, vp],
    "arreau_ve_pbc_reverse": [vp, vp, vp, vp, i32, vp, i32, vp, vp],
    "arreau_d3pm_reverse": [vp, vp, vp, vp, i32, vp, vp, f64, f64, i32, i32, i32, vp, vp],
    "arreau_d3pm_reverse_allowed": [vp, vp, vp, vp, i32, vp, vp, f64, f64, i32, i32, i32, vp, vp, vp, vp],
    "arreau_vp_lattice_reverse_known": [vp, vp, vp, vp, i32, f64, f64, f64, f64, i32, vp, vp, vp, vp, vp],
    "arreau_ve_pbc_reverse_known": [vp, vp, vp, vp, i32, vp, i32, vp, vp, vp, vp],
    "arreau_d3pm_reverse_known": [vp, vp, vp, vp, i32, vp, vp, f64, f64, i32, i32, i32, vp, vp, vp, vp, vp],
    "arreau_step_noise": [C.c_uint64, i32, i32, i32, i32, vp, vp, vp, vp],
    "arreau_sample_init_keyed": [C.c_uint64, i32, i32, vp, vp, vp, f64, vp, vp, vp, vp],
    "arreau_sample_noise_keyed": [C.c_uint64, i32, i32, i32, i32, vp, vp, vp, vp, vp, vp, vp],
    "arreau_denoise_step": [C.POINTER(Weights), C.POINTER(Workspace), C.POINTER(StepArgs), vp],
    "arreau_denoise_step_replay": [C.POINTER(Weights), C.POINTER(Workspace), C.POINTER(StepArgs), C.POINTER(StepReplay), vp],
    # training step
    "arreau_matrix_to_params": [vp, i32, vp, vp, vp],
    "arreau_ve_pbc_forward": [vp, vp, vp, vp, vp, vp, i32, vp, vp, vp],
    "arreau_vp_lattice_forward": [vp, vp, vp, vp, i32, vp, vp],
    "arreau_d3pm_q_sample": [vp, vp, vp, vp, vp, i32, i32, vp, vp],
    "arreau_training_loss": [vp, vp, vp, vp, vp, vp, vp, vp, vp, vp, vp, f64, f64, i32, i32, i32, i32, f64, vp, vp, vp,
                             vp, vp, vp],
    "arreau_eval_noise": [C.c_uint64, i32, i32, i32, i32, vp, vp, vp, vp, vp, vp, vp, vp],
    "arreau_eval_loss": [vp, vp, vp, vp, vp, vp, vp, vp, vp, vp, vp, f64, f64, i32, i32, i32, i32, vp, vp, vp],
    "arreau_train_layout": [i32, i32, i32, C.POINTER(TrainLayout)],
    "arreau_ponita_backward_workspace_bytes": [i32, i64, i32, i32],
    "arreau_ponita_backward": [vp, C.POINTER(TrainLayout), C.POINTER(Weights), C.POINTER(Workspace), vp, vp, vp, vp, vp,
                               vp, vp, vp, vp, vp, vp, i32, i32, f64, vp, vp, vp, vp, i64, vp, i32, i32, vp],
    "arreau_ponita_forward_train": [vp, C.POINTER(TrainLayout), C.POINTER(Weights), C.POINTER(Workspace), vp, vp, vp, vp, vp,
                                    vp, vp, vp, vp, vp, i32, i32, f64, vp, i64, i32, vp, vp, vp, vp],
    "arreau_sgemm": [i32, i32, vp, i64, vp, i64, vp, i64, i32, i32, i64, C.c_float, vp, i32, vp, i64, vp],
    "arreau_fold_basis_w1": [vp, vp, vp, vp, vp],
    "arreau_moments": [vp, vp, i64, vp, vp, vp],
    "arreau_adam_step": [vp, vp, vp, vp, vp, i64, f64, f64, f64, f64, f64, i64, f64, vp, vp, f64, vp],
    # crystal metrics
    "arreau_crystal_metrics": [vp, vp, vp, vp, i32, i32, vp, i32, f64, f64, vp, vp, vp, vp, vp, vp],
    # structure matcher
    "arreau_structure_match": [vp, vp, vp, vp, vp, vp, vp, vp, i32, i32, i32, f64, f64, f64, vp, vp, vp, vp, vp],
    "arreau_structure_fit_pairs": [vp, vp, vp, vp, i32, i32, vp, vp, vp, vp, i32, i32, vp, vp, i32, f64, f64, f64,
                                   vp, vp, vp, vp],
}
RESTYPES = {"arreau_launch_count": i64, "arreau_ponita_backward_workspace_bytes": i64}


def library_path() -> str:
    return _build.LIB_PATH


def load():
    """Load (once) and type the C-ABI library.  Raises if it has not been built."""
    global _lib
    if _lib is not None:
        return _lib
    path = library_path()
    if not os.path.exists(path):
        raise RuntimeError(f"{path} is missing: run `python -m arreau_b200.build` (needs nvcc). "
                           "arreau_b200 has no CPU or PyTorch fallback.")
    lib = C.CDLL(path)
    for name, argtypes in SIGNATURES.items():
        fn = getattr(lib, name)
        fn.argtypes = argtypes
        fn.restype = RESTYPES.get(name, C.c_int)
    _lib = lib
    return lib


def check(rc: int, what: str) -> None:
    if rc == 0:
        return
    if rc < 0:
        raise RuntimeError(f"{what}: {ERRORS.get(rc, rc)}")
    raise RuntimeError(f"{what}: CUDA error {rc}")


def ptr(t):
    """Device (or host) pointer of a torch tensor, None -> NULL."""
    return None if t is None else t.data_ptr()


def call(name: str, *args) -> None:
    check(getattr(load(), name)(*args), name)


def launch_count() -> int:
    return int(load().arreau_launch_count())
