"""ctypes binding of libsmz.so — the C ABI declared in include/smz.h.  Nothing here computes: a
missing or stale library is a hard error (there is no CPU fallback for the search path)."""
import ctypes as C
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "libsmz.so")

SMZ_ABI_VERSION = 2
SMZ_OK, SMZ_E_INVALID_ARG, SMZ_E_CUDA, SMZ_E_CAPACITY, SMZ_E_STATE = 0, -1, -2, -3, -4
NET_EXTERNAL, NET_FP32, NET_BF16, NET_VISION, NET_TC32, NET_F16 = 0, 1, 2, 3, 4, 5
RNG_PHILOX, RNG_TAPE = 0, 1
PATTERN_REFERENCE, PATTERN_PAPER = 0, 1
SEARCH_PUCT, SEARCH_GUMBEL = 0, 1


class smz_config(C.Structure):
    _fields_ = [
        ("abi_version", C.c_int32), ("device", C.c_int32), ("max_trees", C.c_int32),
        ("num_simulations", C.c_int32), ("action_dim", C.c_int32), ("chance_dim", C.c_int32),
        ("max_action_sample", C.c_int32), ("pb_c_base", C.c_int32),
        ("pb_c_init", C.c_double), ("discount", C.c_double), ("root_dirichlet_alpha", C.c_double),
        ("root_exploration_fraction", C.c_double),
        ("obs_dim", C.c_int32), ("state_dim", C.c_int32), ("hidden_dim", C.c_int32),
        ("num_hidden_layers", C.c_int32), ("net_mode", C.c_int32), ("rng_mode", C.c_int32),
        ("lanes_per_tree", C.c_int32), ("record", C.c_int32),
        ("seed", C.c_uint64), ("tree_id_offset", C.c_uint64),
    ]


class smz_dims(C.Structure):
    _fields_ = [
        ("nodes_per_tree", C.c_int32), ("max_children", C.c_int32), ("policy_stride", C.c_int32),
        ("hidden_stride", C.c_int32), ("hidden_slots", C.c_int32), ("path_stride", C.c_int32),
        ("lanes_per_tree", C.c_int32), ("reserved", C.c_int32),
        ("weight_blob_floats", C.c_uint64), ("arena_bytes", C.c_uint64),
    ]


class smz_tree_host(C.Structure):
    _fields_ = [
        ("visit", C.POINTER(C.c_int32)), ("value_sum", C.POINTER(C.c_float)), ("reward", C.POINTER(C.c_float)),
        ("prior", C.POINTER(C.c_float)), ("child_base", C.POINTER(C.c_int32)), ("key", C.POINTER(C.c_int32)),
        ("root_prior", C.POINTER(C.c_double)), ("minmax", C.c_float * 2), ("n_uniforms", C.c_int32),
        ("root_to_play", C.c_int32),
    ]


_P = C.c_void_p
# name -> (restype, argtypes); every symbol include/smz.h declares
SIGNATURES = {
    "smz_create": (C.c_int, [C.POINTER(smz_config), C.POINTER(_P)]),
    "smz_destroy": (C.c_int, [_P]),
    "smz_get_dims": (C.c_int, [_P, C.POINTER(smz_dims)]),
    "smz_last_error": (C.c_char_p, []),
    "smz_set_pbc_table": (C.c_int, [_P, C.POINTER(C.c_double), C.c_int32]),
    "smz_set_player_tables": (C.c_int, [_P, C.POINTER(C.c_int8), C.POINTER(C.c_int32), C.c_int32]),
    "smz_set_weights": (C.c_int, [_P, _P, C.c_uint64, C.c_int32, _P]),
    "smz_set_seed": (C.c_int, [_P, C.c_uint64, C.c_uint64, _P]),
    "smz_set_uniform_tape": (C.c_int, [_P, _P, C.c_int32]),
    "smz_set_node_pattern": (C.c_int, [_P, C.c_int32]),
    "smz_root": (C.c_int, [_P, C.c_int32, _P, _P, _P, C.c_int32, _P, _P]),
    "smz_root_legal": (C.c_int, [_P, C.c_int32, _P, _P, _P, _P, C.c_int32, _P, _P]),
    "smz_set_search": (C.c_int, [_P, C.c_int32, C.c_int32, C.c_double, C.c_double]),
    "smz_sequential_halving_table": (C.c_int, [C.c_int32, _P]),
    "smz_set_root_budgets": (C.c_int, [_P, C.c_int32, _P, _P, _P]),
    "smz_root_gumbel": (C.c_int, [_P, C.c_int32, _P, _P, _P, _P, _P, C.c_int32, _P, _P]),
    "smz_read_gumbel": (C.c_int, [_P, _P, _P, _P, _P]),
    "smz_read_raw_values": (C.c_int, [_P, _P, _P]),
    "smz_simulate": (C.c_int, [_P, C.c_int32, _P]),
    "smz_select": (C.c_int, [_P, C.c_int32, _P, _P, _P, _P]),
    "smz_net_step": (C.c_int, [_P, C.c_int32, _P]),
    "smz_expand_backup": (C.c_int, [_P, C.c_int32, _P, _P, _P, _P]),
    "smz_net_eval": (C.c_int, [_P, C.c_int32, C.c_int32, _P, _P, _P, _P, _P, _P, _P, _P]),
    "smz_backup_select": (C.c_int, [_P, C.c_int32, _P]),
    "smz_read_roots": (C.c_int, [_P, _P, _P, _P, _P, _P, _P]),
    "smz_select_actions": (C.c_int, [_P, C.c_double, _P, _P, _P, _P, _P]),
    "smz_export_tree": (C.c_int, [_P, C.c_int32, C.POINTER(smz_tree_host), _P]),
    "smz_read_hidden": (C.c_int, [_P, C.c_int32, _P, _P]),
    "smz_read_record": (C.c_int, [_P, _P, _P, _P, _P, _P, _P, _P]),
    "smz_stats": (C.c_int, [_P, C.POINTER(C.c_double), C.POINTER(C.c_int64), C.POINTER(C.c_int64), _P]),
}

_lib = None


def load():
    """dlopen libsmz.so and bind every entry point.  Raises if the extension has not been built."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.isfile(LIB_PATH):
        raise RuntimeError(
            f"{LIB_PATH} is missing: build the CUDA extension first (python -c 'import __graft_entry__ as g; "
            "g.build()' or make -C stochastic-muzero_b200/csrc).  There is no CPU fallback.")
    lib = C.CDLL(LIB_PATH)
    for name, (res, args) in SIGNATURES.items():
        fn = getattr(lib, name)      # AttributeError here = header and library out of sync
        fn.restype, fn.argtypes = res, args
    _lib = lib
    return lib
