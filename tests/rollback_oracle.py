"""TEST INFRASTRUCTURE ONLY -- ctypes front-end of tests/rollback_oracle.c: the C oracle with SP-inspired decimation
(tests/sid_oracle.c, included as it is) and conflict rollback, i.e. a step of K_b >= 2 variables that ends in a
unit-propagation conflict is undone and the problem's later steps are halved.

The library is compiled on first use into a temporary directory (keyed by the sources), so the tree stays read-only."""
import ctypes
import hashlib
import os
import subprocess
import tempfile

import numpy as np

from oracle import pdp_oracle as po
from tests import sid_oracle

_HERE = os.path.dirname(os.path.abspath(__file__))
_SRCS = (os.path.join(_HERE, "rollback_oracle.c"), os.path.join(_HERE, "sid_oracle.c"),
         os.path.join(os.path.dirname(_HERE), "oracle", "pdp_oracle.c"))
_lib = None


def lib():
    global _lib
    if _lib is None:
        h = hashlib.sha256()
        for p in _SRCS:
            with open(p, "rb") as f:
                h.update(f.read())
        so = os.path.join(tempfile.gettempdir(), "pdp_rollback_oracle_%s_%d.so" % (h.hexdigest()[:16], os.getuid()))
        if not os.path.exists(so):
            tmp = so + ".%d.tmp" % os.getpid()
            subprocess.check_call(["gcc", "-O2", "-fopenmp", "-fno-fast-math", "-ffp-contract=off", "-shared", "-fPIC",
                                   "-o", tmp, _SRCS[0], "-lm"])
            os.replace(tmp, so)
        L = ctypes.CDLL(so)
        base = sid_oracle.lib()
        for name in ("ora_create", "ora_destroy", "ora_set_state", "ora_set_masks", "ora_get_state", "ora_get_masks",
                     "ora_get_counters", "ora_iters_done", "ora_trace_len", "ora_get_trace", "ora_edge_mask_set",
                     "ora_simplify", "ora_set_variables", "ora_sp_step", "ora_score", "ora_cnf_eval", "ora_energy",
                     "ora_energy_diff", "ora_compute_edge_mask", "ora_iterate", "ora_run", "ora_count_active_variables",
                     "ora_random_fill", "ora_local_search", "ora_deduplicate", "ora_num_threads", "ora_set_math_mode",
                     "sid_iterate", "sid_run", "sid_decimation_select"):
            src, dst = getattr(base, name), getattr(L, name)
            dst.restype, dst.argtypes = src.restype, src.argtypes
        P, I64, F32, I = ctypes.c_void_p, ctypes.c_int64, ctypes.c_float, ctypes.c_int
        L.rb_create.restype = P
        L.rb_create.argtypes = [P]
        L.rb_destroy.restype = None
        L.rb_destroy.argtypes = [P]
        L.rb_set.restype = None
        L.rb_set.argtypes = [P, I]
        L.rb_get.restype = None
        L.rb_get.argtypes = [P, P, P, P]
        L.rb_iterate.restype = I64
        L.rb_iterate.argtypes = [P, P, F32, F32, I, I, F32, F32]
        L.rb_run.restype = I64
        L.rb_run.argtypes = [P, P, I64, F32, F32, I, I, F32, F32]
        _lib = L
    return _lib


def set_math_mode(correctly_rounded):
    """this library's copy of the oracle's math mode"""
    lib().ora_set_math_mode(1 if correctly_rounded else 0)


class RollbackOracle(sid_oracle.SidOracle):
    """SidOracle whose loop undoes a K_b >= 2 step that ends in a unit-propagation conflict (set_conflict_rollback) and
    halves the problem's later steps; strict = 0 only"""

    def __init__(self, graph_map, batch_variable_map, batch_function_map, edge_feature, batch_size=None):
        L = lib()
        self.strict = False
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
        self._h = L.ora_create(self.E, self.V, self.F, self.B, po._p(gm), po._p(sign), po._p(self.bvm), po._p(self.bfm), 0)
        self._L = L
        self._rb = L.rb_create(self._h)

    def __del__(self):
        try:
            if getattr(self, "_rb", None):
                self._L.rb_destroy(self._rb)
                self._rb = None
        except Exception:
            pass
        super(RollbackOracle, self).__del__()

    def set_conflict_rollback(self, on):
        self._L.rb_set(self._rb, 1 if on else 0)

    def rollbacks(self):
        """(h [B], r [B], iteration of the last rollback [B], 0 = none), int64"""
        h, r, last = (np.zeros(self.B, np.int64) for _ in range(3))
        self._L.rb_get(self._rb, po._p(h), po._p(r), po._p(last))
        return h, r, last

    def iterate(self, tol, t_max, check_termination=True, batch_replication=1, pi=0.0):
        return int(self._L.rb_iterate(self._h, self._rb, tol, t_max, 1 if check_termination else 0, batch_replication, pi,
                                      self.fraction))

    def run(self, T, tol, t_max, check_termination=True, batch_replication=1, pi=0.0):
        return int(self._L.rb_run(self._h, self._rb, T, tol, t_max, 1 if check_termination else 0, batch_replication, pi,
                                  self.fraction))
