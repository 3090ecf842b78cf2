"""ctypes binding of the C ABI declared in include/pct_b200.h (libpct_b200.so, built in-tree by csrc/Makefile).

The library is the product: if it is missing this module raises — there is no Python / CPU fallback."""
import ctypes as C
import os
import subprocess

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("PCT_B200_LIB", os.path.join(_HERE, "libpct_b200.so"))  # env override: tuning experiments only

PCT_DISCRETE, PCT_CONTINUOUS = 0, 1
PCT_F32, PCT_F64 = 0, 1
PCT_ITEMS_RANDOM, PCT_ITEMS_STREAM = 0, 1
FLAG_NAMES = {1: "box_overflow", 2: "bad_action", 4: "ems_overflow", 8: "cand_overflow", 16: "edge_overflow", 32: "support_overflow",
              64: "sync_timeout"}


class Config(C.Structure):
    _fields_ = [("domain", C.c_int32), ("setting", C.c_int32), ("container_size", C.c_double * 3),
                ("internal_node_holder", C.c_int32), ("leaf_node_holder", C.c_int32), ("obs_dtype", C.c_int32),
                ("item_mode", C.c_int32), ("size_minimum", C.c_double), ("sample_from_distribution", C.c_int32),
                ("sample_left_bound", C.c_double), ("sample_right_bound", C.c_double), ("seed", C.c_uint64),
                ("env_id_base", C.c_int64), ("no_auto_reset", C.c_int32), ("lnes", C.c_int32), ("shuffle", C.c_int32)]


LNES_CODES = {"EMS": 0, "EV": 1, "EP": 2, "CP": 3, "FC": 4}
HEURISTIC_CODES = {"LSAH": 0, "OnlineBPH": 1, "BR": 2, "MACS": 3, "DBL": 4, "HM": 5, "RANDOM": 6}  # heuristic.py:593-606 names


class StepInfo(C.Structure):
    _fields_ = [("counter", C.c_int32), ("flags", C.c_int32), ("ratio", C.c_float), ("ep_reward", C.c_float),
                ("ep_len", C.c_int32), ("n_leaf", C.c_int32), ("n_cand", C.c_int32), ("n_ems", C.c_int32)]


class StateDump(C.Structure):
    _fields_ = [("n_boxes", C.c_int32), ("n_ems", C.c_int32), ("n_leaf", C.c_int32), ("flags", C.c_int32),
                ("draw_pos", C.c_int64), ("next_box", C.c_double * 3), ("next_den", C.c_double),
                ("boxes", (C.c_double * 7) * 80), ("ems", (C.c_double * 6) * 256)]


EXPORTS = ["pct_create", "pct_destroy", "pct_last_error", "pct_set_item_set", "pct_set_item_stream", "pct_set_trajectory_length", "pct_reset", "pct_step",
           "pct_step_host", "pct_reset_host", "pct_policy_random", "pct_policy_random_dev", "pct_get_state", "pct_obs_len", "pct_num_envs",
           "pct_state_bytes_per_env", "pct_kernel_launches", "pct_version", "pct_profile_enable", "pct_profile_read", "pct_heuristic_actions",
           "pct_heuristic_actions_f64", "pct_query_placement", "pct_query_placement_f64", "pct_env_record_bytes", "pct_save_envs", "pct_load_envs"]
RECORD_STATUS = {1: "not a record of this configuration", 2: "item-stream row not in this handle", 3: "env id out of range"}  # pct_load_envs


def build(verbose=False):
    """Compile csrc/*.cu for sm_100a into libpct_b200.so (nvcc cross-compiles without a GPU)."""
    subprocess.check_call(["make", "-C", os.path.join(_HERE, "csrc")] + ([] if verbose else ["-s"]))
    return LIB_PATH


_lib = None


def lib():
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise RuntimeError("pct_b200: %s is missing — run `python -c 'import __graft_entry__ as g; g.build()'` "
                           "(there is no CPU fallback)" % LIB_PATH)
    L = C.CDLL(LIB_PATH)
    vp, i32, i64, u64 = C.c_void_p, C.c_int32, C.c_int64, C.c_uint64
    L.pct_create.argtypes = [C.POINTER(Config), i32, i32, C.POINTER(vp)]
    L.pct_destroy.argtypes = [vp]
    L.pct_destroy.restype = None
    L.pct_last_error.argtypes = [vp]
    L.pct_last_error.restype = C.c_char_p
    L.pct_set_item_set.argtypes = [vp, C.POINTER(C.c_double), i32]
    L.pct_set_item_stream.argtypes = [vp, C.POINTER(C.c_double), i32]
    L.pct_set_trajectory_length.argtypes = [vp, i32]
    L.pct_reset.argtypes = [vp, vp, vp]
    L.pct_step.argtypes = [vp, vp, i32, vp, vp, vp, vp, vp, vp]
    L.pct_step_host.argtypes = [vp, vp, i32, vp, vp, vp, vp, vp]
    L.pct_reset_host.argtypes = [vp, vp]
    L.pct_policy_random.argtypes = [vp, vp, u64, i64, vp]
    L.pct_policy_random_dev.argtypes = [vp, vp, u64, vp, vp]
    L.pct_get_state.argtypes = [vp, i32, C.POINTER(StateDump)]
    L.pct_obs_len.argtypes = [vp]
    L.pct_num_envs.argtypes = [vp]
    L.pct_state_bytes_per_env.argtypes = [vp]
    L.pct_state_bytes_per_env.restype = i64
    L.pct_kernel_launches.argtypes = [vp]
    L.pct_kernel_launches.restype = i64
    L.pct_version.restype = C.c_char_p
    L.pct_profile_enable.argtypes = [vp, i32]
    L.pct_profile_read.argtypes = [vp, C.POINTER(C.c_double), C.POINTER(i32)]
    L.pct_heuristic_actions.argtypes = [vp, i32, vp, u64, i64, vp]
    L.pct_heuristic_actions_f64.argtypes = [vp, i32, vp, vp]
    L.pct_query_placement.argtypes = [vp, i32, C.POINTER(i32), i32, i32, C.c_double, C.POINTER(i32), C.POINTER(i32), C.POINTER(i32)]
    L.pct_query_placement_f64.argtypes = [vp, i32, C.POINTER(C.c_double), C.c_double, C.c_double, C.c_double, C.POINTER(i32),
                                          C.POINTER(C.c_double)]
    L.pct_env_record_bytes.argtypes = [vp]
    L.pct_env_record_bytes.restype = i64
    L.pct_save_envs.argtypes = [vp, vp, i32, vp, vp]
    L.pct_load_envs.argtypes = [vp, vp, i32, vp, vp, vp, vp]
    _lib = L
    return L
