"""ctypes binding of libpdp_b200.so (the C ABI declared in include/pdp_b200.h).

There is no CPU fallback: if the shared library is missing or a call fails, an exception is raised.
"""
import ctypes
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "csrc", "libpdp_b200.so")
# TEST build with correctly rounded fp32 log/exp (bitwise comparisons against the C oracle)
STRICT_LIB_PATH = os.path.join(_HERE, "csrc", "libpdp_b200_strict.so")

_libs = {}

P = ctypes.c_void_p
I32 = ctypes.c_int32
I64 = ctypes.c_int64
U64 = ctypes.c_uint64
F32 = ctypes.c_float


class SpParams(ctypes.Structure):
    """mirror of pdp_sp_params (include/pdp_b200.h)"""
    _fields_ = [("iterations", I32), ("tolerance", F32), ("t_max", I32), ("pi", F32),
                ("check_termination", I32), ("batch_replication", I32), ("full_state", I32), ("flags", I32)]


# name -> (restype, argtypes); every symbol include/pdp_b200.h declares
SIGNATURES = {
    "pdp_version": (ctypes.c_char_p, []),
    "pdp_last_error": (ctypes.c_char_p, []),
    "pdp_workspace_bytes": (ctypes.c_size_t, [I64, I64, I64, I64]),
    "pdp_create": (ctypes.c_int, [ctypes.POINTER(P), P, P, P, P, I64, I64, I64, I64, P, ctypes.c_size_t, P]),
    "pdp_destroy": (ctypes.c_int, [P]),
    "pdp_reset": (ctypes.c_int, [P, P]),
    "pdp_cnf_eval": (ctypes.c_int, [P, P, P, P, P]),
    "pdp_cnf_eval_edges_scratch_bytes": (ctypes.c_size_t, [I64, I64]),
    "pdp_cnf_eval_edges": (ctypes.c_int, [P, P, P, I64, I64, I64, I64, P, P, P, P, P]),
    "pdp_energy": (ctypes.c_int, [P, P, P, P, P, P, P]),
    "pdp_energy_diff": (ctypes.c_int, [P, P, P, P, P, P]),
    "pdp_sp_step": (ctypes.c_int, [P, P, P, P, P, P, P, F32, P, P, P]),
    "pdp_sp_step_adapted": (ctypes.c_int, [P, P, P, P, P, P, P, P, F32, P, P, P]),
    "pdp_edge_aggregate": (ctypes.c_int, [P, I32, P, I32, P, P, P]),
    "pdp_edge_mlp_forward": (ctypes.c_int, [P, I32, P, I32, P, I32, I64, P, P, I32, I32, I32, I32, I32, P, P, P]),
    "pdp_edge_nn_chunk_k": (ctypes.c_int, []),
    "pdp_edge_nn_swizzle": (ctypes.c_int, []),
    "pdp_edge_gru_forward": (ctypes.c_int, [P, I32, P, I32, P, I32, I64, P, P, I32, I32, I32, P, P, P]),
    "pdp_score": (ctypes.c_int, [P, P, P, F32, P, P]),
    "pdp_load_state": (ctypes.c_int, [P, P, P, P, P, P]),
    "pdp_load_state_const": (ctypes.c_int, [P, F32, F32, F32, F32, F32, P]),
    "pdp_store_state": (ctypes.c_int, [P, P, P, P]),
    "pdp_set_masks": (ctypes.c_int, [P, P, P, P, P]),
    "pdp_get_masks": (ctypes.c_int, [P, P, P, P, P, P, P, P]),
    "pdp_set_active": (ctypes.c_int, [P, P, P]),
    "pdp_get_problem_flags": (ctypes.c_int, [P, P, P, P, P]),
    "pdp_simplify": (ctypes.c_int, [P, P]),
    "pdp_set_variables": (ctypes.c_int, [P, P, P]),
    "pdp_sp_run": (ctypes.c_int, [P, ctypes.POINTER(SpParams), P, P]),
    "pdp_count_active_variables": (ctypes.c_int, [P, ctypes.POINTER(I64), P]),
    "pdp_random_fill": (ctypes.c_int, [P, P, P]),
    "pdp_walksat": (ctypes.c_int, [P, I32, F32, I32, P, P, U64, P, P, P]),
    "pdp_deduplicate": (ctypes.c_int, [P, I32, P, P, P, P]),
    "pdp_set_decimation_fraction": (ctypes.c_int, [P, F32]),
    "pdp_decimation_select": (ctypes.c_int, [P, P, P, P, F32, P, P]),
    "pdp_rollback_scratch_bytes": (ctypes.c_size_t, [I64, I64, I64]),
    "pdp_set_conflict_rollback": (ctypes.c_int, [P, P, ctypes.c_size_t]),
    "pdp_set_reinforce": (ctypes.c_int, [P, P, I32, F32]),
    "pdp_get_rollbacks": (ctypes.c_int, [P, P, P, P]),
    "pdp_debug_check_edge_mask": (ctypes.c_int, [P, P, P]),
    "pdp_set_trace_buffer": (ctypes.c_int, [P, P, I32]),
    "pdp_trace_length": (ctypes.c_int, [P, ctypes.POINTER(I32), P]),
    "pdp_debug_check_layout": (ctypes.c_int, [P, P, ctypes.POINTER(I32 * 5), P]),
    "pdp_launch_count": (I64, [P]),
    "pdp_host_parse_ints": (I64, [ctypes.c_char_p, I64, P, I64]),
    "pdp_host_parse_rows": (I64, [ctypes.c_char_p, I64, P, P, I64, P, P, P, P, I64]),
    "pdp_host_parse_dimacs": (ctypes.c_int, [ctypes.c_char_p, I64, P, I64, ctypes.POINTER(I64 * 4)]),
}


class PdpError(RuntimeError):
    pass


def load(strict_math=False):
    """Loads the shared library; raises if it has not been built (python __graft_entry__.py build).
    strict_math=True loads the test build (tests only)."""
    key = bool(strict_math)
    if key in _libs:
        return _libs[key]
    path = STRICT_LIB_PATH if key else os.environ.get("PDP_B200_LIB", LIB_PATH)   # override: A/B builds of the product library
    if not os.path.exists(path):
        raise PdpError("%s not found -- build it with pdp_solver_b200/csrc/build.sh "
                       "(there is no CPU fallback)" % path)
    lib = ctypes.CDLL(path)
    for name, (res, args) in SIGNATURES.items():
        fn = getattr(lib, name)   # AttributeError if the symbol is missing: fail loudly
        fn.restype = res
        fn.argtypes = args
    _libs[key] = lib
    return lib


def check(rc, what="", lib=None):
    if rc != 0:
        msg = (lib or load()).pdp_last_error()
        raise PdpError("%s failed (%d): %s" % (what, rc, msg.decode() if msg else "?"))
