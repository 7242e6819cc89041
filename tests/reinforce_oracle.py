"""TEST INFRASTRUCTURE ONLY -- ctypes front-end of tests/reinforce_oracle.c: the C oracle (oracle/pdp_oracle.c, included as
it is) with the loop of model type `reinforce` as the library's persistent kernel runs it (pdp_set_reinforce).

The library is compiled on first use into a temporary directory (keyed by the sources), so the tree stays read-only."""
import ctypes
import hashlib
import os
import subprocess
import tempfile

import numpy as np

from oracle import pdp_oracle as po

_HERE = os.path.dirname(os.path.abspath(__file__))
_SRC = os.path.join(_HERE, "reinforce_oracle.c")
_ORACLE_SRC = os.path.join(os.path.dirname(_HERE), "oracle", "pdp_oracle.c")
_lib = None


def lib():
    global _lib
    if _lib is None:
        h = hashlib.sha256()
        for p in (_SRC, _ORACLE_SRC):
            with open(p, "rb") as f:
                h.update(f.read())
        so = os.path.join(tempfile.gettempdir(), "pdp_reinforce_oracle_%s_%d.so" % (h.hexdigest()[:16], os.getuid()))
        if not os.path.exists(so):
            tmp = so + ".%d.tmp" % os.getpid()
            subprocess.check_call(["gcc", "-O2", "-fopenmp", "-fno-fast-math", "-ffp-contract=off", "-shared", "-fPIC",
                                   "-o", tmp, _SRC, "-lm"])
            os.replace(tmp, so)
        L = ctypes.CDLL(so)
        base = po.lib()
        for name in ("ora_create", "ora_destroy", "ora_set_state", "ora_set_masks", "ora_get_state", "ora_get_masks",
                     "ora_simplify", "ora_cnf_eval", "ora_set_math_mode"):
            src, dst = getattr(base, name), getattr(L, name)
            dst.restype, dst.argtypes = src.restype, src.argtypes
        P, I64, F32, I = ctypes.c_void_p, ctypes.c_int64, ctypes.c_float, ctypes.c_int
        L.rf_run.restype = I64
        L.rf_run.argtypes = [P, I64, F32, F32, P, I, I, P, P]
        _lib = L
    return _lib


def set_math_mode(correctly_rounded):
    """this library's copy of the oracle's math mode (oracle.pdp_oracle.set_math_mode sets the other library's)"""
    lib().ora_set_math_mode(1 if correctly_rounded else 0)


class ReinforceOracle(po.Oracle):
    """po.Oracle (strict = 0: every problem as in a batch of one) with the reinforce loop"""

    def __init__(self, graph_map, batch_variable_map, batch_function_map, edge_feature, batch_size=None):
        L = lib()
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

    def reinforce_run(self, init_prop, init_dec, T, pi, p_dec, coins, check_termination=True, batch_replication=1):
        """simplify, load the state, run.  Returns (iterations, merged prediction [iterations, V] (with
        check_termination), freeze iteration per problem [B] (-1: never retired), final q [E,3], final [eta, ext] [E,2])"""
        self.simplify()
        self.set_state(init_prop, init_dec)
        c = po._f32(np.asarray(coins).reshape(-1))
        assert c.shape[0] >= int(T)
        merged = np.zeros((max(int(T), 1), self.V), np.float32)
        freeze = np.empty(self.B, np.int32)
        n = int(self._L.rf_run(self._h, int(T), float(pi), float(p_dec), po._p(c), 1 if check_termination else 0,
                               int(batch_replication), po._p(merged), po._p(freeze)))
        q, f = self.state()
        return n, merged[:n], freeze, q, f
