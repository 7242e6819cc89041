"""TEST INFRASTRUCTURE ONLY -- ctypes front-end of tests/sid_oracle.c: the C oracle (oracle/pdp_oracle.c, included as it
is) with SP-inspired decimation, i.e. a fraction of each problem's active variables fixed per decimation step.

The library is compiled on first use into a temporary directory (keyed by the sources), so the tree stays read-only."""
import ctypes
import hashlib
import math
import os
import subprocess
import tempfile

import numpy as np

from oracle import pdp_oracle as po

_HERE = os.path.dirname(os.path.abspath(__file__))
_SRC = os.path.join(_HERE, "sid_oracle.c")
_ORACLE_SRC = os.path.join(os.path.dirname(_HERE), "oracle", "pdp_oracle.c")
_lib = None


def lib():
    global _lib
    if _lib is None:
        h = hashlib.sha256()
        for p in (_SRC, _ORACLE_SRC):
            with open(p, "rb") as f:
                h.update(f.read())
        so = os.path.join(tempfile.gettempdir(), "pdp_sid_oracle_%s_%d.so" % (h.hexdigest()[:16], os.getuid()))
        if not os.path.exists(so):
            tmp = so + ".%d.tmp" % os.getpid()
            subprocess.check_call(["gcc", "-O2", "-fopenmp", "-fno-fast-math", "-ffp-contract=off", "-shared", "-fPIC",
                                   "-o", tmp, _SRC, "-lm"])
            os.replace(tmp, so)
        L = ctypes.CDLL(so)
        base = po.lib()
        # the oracle's own entry points: the same signatures as oracle/pdp_oracle.py declares
        for name in ("ora_create", "ora_destroy", "ora_set_state", "ora_set_masks", "ora_get_state", "ora_get_masks",
                     "ora_get_counters", "ora_iters_done", "ora_trace_len", "ora_get_trace", "ora_edge_mask_set",
                     "ora_simplify", "ora_set_variables", "ora_sp_step", "ora_score", "ora_cnf_eval", "ora_energy",
                     "ora_energy_diff", "ora_compute_edge_mask", "ora_iterate", "ora_run", "ora_count_active_variables",
                     "ora_random_fill", "ora_local_search", "ora_deduplicate", "ora_num_threads", "ora_set_math_mode"):
            src, dst = getattr(base, name), getattr(L, name)
            dst.restype, dst.argtypes = src.restype, src.argtypes
        P, I64, F32, I = ctypes.c_void_p, ctypes.c_int64, ctypes.c_float, ctypes.c_int
        L.sid_iterate.restype = I64
        L.sid_iterate.argtypes = [P, F32, F32, I, I, F32, F32]
        L.sid_run.restype = I64
        L.sid_run.argtypes = [P, I64, F32, F32, I, I, F32, F32]
        L.sid_decimation_select.restype = I
        L.sid_decimation_select.argtypes = [P, P, P, P, F32, P]
        _lib = L
    return _lib


def check_fraction(fraction, strict=False):
    f = float(fraction)
    if not (math.isfinite(f) and 0.0 <= f < 1.0) or (strict and f > 0.0):
        raise ValueError("decimation fraction %r: must be finite, 0 <= f < 1, and 0 on a strict oracle" % (fraction,))
    return f


def set_math_mode(correctly_rounded):
    """this library's copy of the oracle's math mode (oracle.pdp_oracle.set_math_mode sets the other library's)"""
    lib().ora_set_math_mode(1 if correctly_rounded else 0)


class SidOracle(po.Oracle):
    """po.Oracle whose loop decimates a fraction of each selected problem's active variables per step
    (set_decimation_fraction; 0, the default, is the oracle's own arg-max rule)"""

    def __init__(self, graph_map, batch_variable_map, batch_function_map, edge_feature, strict=False, batch_size=None):
        L = lib()
        self.strict = bool(strict)
        self.fraction = 0.0
        gm = np.ascontiguousarray(np.asarray(graph_map, dtype=np.int32))
        self.E = int(gm.shape[1])
        self.gm = gm
        self.bvm = np.ascontiguousarray(np.asarray(batch_variable_map, dtype=np.int32))
        self.bfm = np.ascontiguousarray(np.asarray(batch_function_map, dtype=np.int32))
        self.V = int(self.bvm.shape[0])
        self.F = int(self.bfm.shape[0])
        if batch_size is None:
            batch_size = int(self.bvm.max()) + 1 if self.V > 0 else 0
        self.B = int(batch_size)
        sign = po._f32(np.asarray(edge_feature).reshape(-1))
        self._h = L.ora_create(self.E, self.V, self.F, self.B, po._p(gm), po._p(sign), po._p(self.bvm), po._p(self.bfm),
                               1 if strict else 0)
        self._L = L

    def set_decimation_fraction(self, fraction):
        self.fraction = check_fraction(fraction, self.strict)

    def iterate(self, tol, t_max, check_termination=True, batch_replication=1, pi=0.0):
        return int(self._L.sid_iterate(self._h, tol, t_max, 1 if check_termination else 0, batch_replication, pi, self.fraction))

    def run(self, T, tol, t_max, check_termination=True, batch_replication=1, pi=0.0):
        return int(self._L.sid_run(self._h, T, tol, t_max, 1 if check_termination else 0, batch_replication, pi, self.fraction))

    def decimation_select(self, coeff, score, fraction, problem_sel=None):
        """the rule on given coefficients [V] / scores [V] (pdp_decimation_select): sign(score) on the taken variables"""
        f = check_fraction(fraction, self.strict)
        c, sc = po._f32(np.asarray(coeff).reshape(-1)), po._f32(np.asarray(score).reshape(-1))
        ps = None if problem_sel is None else np.ascontiguousarray(np.asarray(problem_sel, dtype=np.uint8).reshape(-1))
        out = np.empty(self.V, np.float32)
        if self._L.sid_decimation_select(self._h, po._p(c), po._p(sc), po._p(ps), f, po._p(out)) != 0:
            raise ValueError("decimation fraction %r rejected" % (fraction,))
        return out
