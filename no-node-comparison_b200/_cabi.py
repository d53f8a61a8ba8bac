"""ctypes declarations of include/nbody_b200.h (shared by the product loader and the test harness)."""
from __future__ import annotations

import ctypes as C

c_f = C.c_void_p  # device (or, under the test emulator, host) pointers travel as void*


class NbEgnoConfig(C.Structure):
    _fields_ = [("B", C.c_int32), ("N", C.c_int32), ("T", C.c_int32), ("n_layers", C.c_int32),
                ("num_modes", C.c_int32), ("in_node_nf", C.c_int32), ("in_edge_nf", C.c_int32),
                ("time_emb_dim", C.c_int32), ("use_time_conv", C.c_int32), ("num_inputs", C.c_int32)]


class NbSegnoConfig(C.Structure):
    _fields_ = [("B", C.c_int32), ("N", C.c_int32), ("T", C.c_int32), ("in_node_nf", C.c_int32),
                ("in_edge_nf", C.c_int32), ("recurrent", C.c_int32), ("coords_weight", C.c_float),
                ("h_given", C.c_int32)]


EXPORTS = {
    "nb_version": (C.c_int, []),
    "nb_last_error": (C.c_char_p, []),
    "nb_egno_param_count": (C.c_int64, [C.POINTER(NbEgnoConfig)]),
    "nb_segno_param_count": (C.c_int64, [C.POINTER(NbSegnoConfig)]),
    "nb_egno_saved_floats": (C.c_int64, [C.POINTER(NbEgnoConfig)]),
    "nb_egno_workspace_floats": (C.c_int64, [C.POINTER(NbEgnoConfig), C.c_int]),
    "nb_segno_saved_floats": (C.c_int64, [C.POINTER(NbSegnoConfig)]),
    "nb_segno_workspace_floats": (C.c_int64, [C.POINTER(NbSegnoConfig), C.c_int]),
    "nb_egno_forward": (C.c_int, [C.POINTER(NbEgnoConfig)] + [c_f] * 14),
    "nb_egno_backward": (C.c_int, [C.POINTER(NbEgnoConfig)] + [c_f] * 15),
    "nb_segno_forward": (C.c_int, [C.POINTER(NbSegnoConfig)] + [c_f] * 11),
    "nb_segno_backward": (C.c_int, [C.POINTER(NbSegnoConfig)] + [c_f] * 13),
    "nb_egno_input_grad_workspace_floats": (C.c_int64, [C.POINTER(NbEgnoConfig)]),
    "nb_egno_backward_ex": (C.c_int, [C.POINTER(NbEgnoConfig)] + [c_f] * 19),
    "nb_egno_forward_ft": (C.c_int, [C.POINTER(NbEgnoConfig)] + [c_f] * 14),
    "nb_egno_backward_ft": (C.c_int, [C.POINTER(NbEgnoConfig)] + [c_f] * 21),
    "nb_segno_input_grad_workspace_floats": (C.c_int64, [C.POINTER(NbSegnoConfig)]),
    "nb_segno_backward_ex": (C.c_int, [C.POINTER(NbSegnoConfig)] + [c_f] * 16),
    "nb_segno_embed_forward": (C.c_int, [C.POINTER(NbSegnoConfig), c_f, C.c_int64, c_f, c_f, c_f]),
    "nb_segno_embed_backward_workspace_floats": (C.c_int64, [C.POINTER(NbSegnoConfig), C.c_int64]),
    "nb_segno_embed_backward": (C.c_int, [C.POINTER(NbSegnoConfig), C.c_int64] + [c_f] * 5),
    "nb_segno_merge_forward": (C.c_int, [C.c_int32, C.c_int64, C.c_int32, C.c_int32] + [c_f] * 12),
    "nb_segno_merge_backward_workspace_floats": (C.c_int64, [C.c_int64]),
    "nb_segno_merge_backward": (C.c_int, [C.c_int32, C.c_int64, C.c_int32, C.c_int32] + [c_f] * 18 + [C.c_int32, c_f, c_f]),
    "nb_accumulate": (C.c_int, [C.c_int64, c_f, c_f, c_f]),
    "nb_check_canonical_edges": (C.c_int, [c_f, c_f, C.c_int64, C.c_int32, C.c_int32, c_f, c_f]),
    "nb_egcl_edge_forward": (C.c_int, [C.c_int32] * 5 + [c_f] * 5 + [C.c_int32] * 3 + [c_f] * 9),
    "nb_egcl_edge_backward_workspace_floats": (C.c_int64, [C.c_int32, C.c_int32]),
    "nb_egcl_edge_backward": (C.c_int, [C.c_int32] * 5 + [c_f] * 5 + [C.c_int32] * 3 + [c_f] * 14),
    "nb_nbody_features": (C.c_int, [C.c_int32] * 3 + [c_f] * 8),
    "nb_nbody_energy": (C.c_int, [C.c_int32] * 4 + [C.c_float] + [c_f] * 5),
    "nb_sim_charged": (C.c_int, [C.c_int32] * 4 + [C.c_double] * 4 + [c_f] * 6),
    "nb_sim_gravity": (C.c_int, [C.c_int32] * 4 + [C.c_double] * 3 + [c_f] * 7),
    "nb_traj_mse_workspace_floats": (C.c_int64, [C.c_int32]),
    "nb_traj_mse": (C.c_int, [C.c_int32, C.c_int64, C.c_int32, C.c_int32] + [c_f] * 7),
    "nb_adam_step": (C.c_int, [C.c_int64] + [c_f] * 5 + [C.c_int32] + [C.c_double] * 6 + [c_f]),
    "nb_adam_step_peers": (C.c_int, [C.c_int64, c_f, C.POINTER(C.c_void_p), C.c_int32] + [c_f] * 3 + [C.c_int32] + [C.c_double] * 6 + [c_f]),
    "nb_launch_count": (C.c_longlong, []),
    "nb_profile_enable": (C.c_int, [C.c_int]),
    "nb_profile_read": (C.c_int, [C.POINTER(C.c_double), C.POINTER(C.c_longlong)]),
    "nb_set_edge_impl": (C.c_int, [C.c_int]),
    "nb_set_node_impl": (C.c_int, [C.c_int]),
    "nb_get_node_impl": (C.c_int, []),
    "nb_set_node_fused": (C.c_int, [C.c_int]),
    "nb_get_node_fused": (C.c_int, []),
    "nb_set_segno_fused": (C.c_int, [C.c_int]),
    "nb_get_segno_fused": (C.c_int, []),
    "nb_get_edge_impl": (C.c_int, []),
    "nb_set_edge_fwd3": (C.c_int, [C.c_int]),
    "nb_get_edge_fwd3": (C.c_int, []),
    "nb_tc_selftest": (C.c_int, [C.c_int32, c_f, c_f, c_f, c_f]),
    "nb_silu_selftest": (C.c_int, [C.c_int64, c_f, c_f, c_f, c_f]),
}


def declare(lib: C.CDLL) -> C.CDLL:
    """Attach restype/argtypes for every symbol the header declares; raises if one is missing."""
    for name, (res, args) in EXPORTS.items():
        fn = getattr(lib, name)  # AttributeError -> missing export
        fn.restype = res
        fn.argtypes = args
    return lib
