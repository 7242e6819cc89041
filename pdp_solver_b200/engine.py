"""Device context: one batch of CNFs resident on a B200, driven through the C ABI of libpdp_b200.so.

PyTorch is only plumbing here (device memory, streams); all arithmetic happens in the library's CUDA
kernels.  There is no fallback path: without a CUDA device or without the built library every call
raises.
"""
import ctypes
import os

import torch

from . import _lib
from ._lib import P, SpParams


def _ptr(t):
    return None if t is None else ctypes.c_void_p(t.data_ptr())


def _stream():
    return ctypes.c_void_p(torch.cuda.current_stream().cuda_stream)


def _on_own_device(cls):
    """Every public method of Context runs with the context's device current (the library launches on the current
    device, on torch's current stream of that device): a context may be used while another GPU is current, e.g. by the
    per-device worker threads of the multi-GPU predict path."""
    import functools

    def wrap(fn):
        @functools.wraps(fn)
        def inner(self, *a, **k):
            if torch.cuda.current_device() == self.device.index:
                return fn(self, *a, **k)
            with torch.cuda.device(self.device):
                return fn(self, *a, **k)
        return inner

    for name, fn in list(vars(cls).items()):
        if callable(fn) and not name.startswith("_"):
            setattr(cls, name, wrap(fn))
    return cls


def _f32(t, device):
    if t is None:
        return None
    return t.to(device=device, dtype=torch.float32).contiguous()


def check(rc, what=""):
    _lib.check(rc, what)


@_on_own_device
class Context(object):
    """Factor graph of a batch + the mutable solver state (SATProblem and SequentialDecimator state of the
    reference, pdp/nn/solver.py:19-54 and pdp/nn/pdp_decimate.py:109-120)."""

    def __init__(self, graph_map, batch_variable_map, batch_function_map, edge_feature, batch_size=None,
                 strict_math=False):
        if not torch.cuda.is_available():
            raise _lib.PdpError("pdp_solver_b200 needs a CUDA device (sm_100a); there is no CPU fallback")
        self._L = _lib.load(strict_math)   # strict_math: the test build, see csrc/build.sh
        dev = graph_map.device
        if dev.type != "cuda":
            raise _lib.PdpError("Context expects CUDA tensors (got %s)" % dev)
        self.device = dev
        self._gm = graph_map.to(torch.int32).contiguous()
        self._bvm = batch_variable_map.to(torch.int32).contiguous()
        self._bfm = batch_function_map.to(torch.int32).contiguous()
        self._ef = edge_feature.to(torch.float32).reshape(-1).contiguous()
        self.E = int(self._gm.shape[1])
        self.V = int(self._bvm.shape[0])
        self.F = int(self._bfm.shape[0])
        if batch_size is None:
            batch_size = int(self._bvm.max().item()) + 1 if self.V > 0 else 0   # solver.py:53
        self.B = int(batch_size)
        with torch.cuda.device(dev):
            nbytes = self._L.pdp_workspace_bytes(self.E, self.V, self.F, self.B)
            self._ws = torch.empty(nbytes, dtype=torch.uint8, device=dev)
            h = P()
            self._check(self._L.pdp_create(ctypes.byref(h), _ptr(self._gm), _ptr(self._ef), _ptr(self._bvm), _ptr(self._bfm),
                                     self.E, self.V, self.F, self.B, _ptr(self._ws), nbytes, _stream()), "pdp_create")
        self._h = h
        self._iters = torch.zeros(2, dtype=torch.int32, device=dev)
        self._trace = None
        # optional CUDA-event timing of the two persistent kernels (bench.py's roofline numbers)
        self._events = {} if os.environ.get("PDP_B200_TIMING") == "1" else None

    def _check(self, rc, what=""):
        _lib.check(rc, what, self._L)

    def _timed(self, name, fn):
        if self._events is None:
            return fn()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        r = fn()
        e1.record()
        self._events.setdefault(name, []).append((e0, e1))
        return r

    @property
    def timing(self):
        """name -> total milliseconds (synchronises); None unless PDP_B200_TIMING=1"""
        if self._events is None:
            return None
        torch.cuda.synchronize(self.device)
        return {k: sum(a.elapsed_time(b) for a, b in v) for k, v in self._events.items()}

    def __del__(self):
        try:
            if getattr(self, "_h", None):
                self._L.pdp_destroy(self._h)
                self._h = None
        except Exception:
            pass

    # ------------------------------------------------------------------------------------------
    def _new(self, *shape, dtype=torch.float32):
        return torch.empty(*shape, dtype=dtype, device=self.device)

    def reset(self):
        self._check(self._L.pdp_reset(self._h, _stream()), "pdp_reset")

    def check_layout(self):
        """(errors int32[8] on the host, info dict) of the blocked message layout self-check (tests)"""
        errs = self._new(8, dtype=torch.int32)
        info = (ctypes.c_int32 * 5)()
        self._check(self._L.pdp_debug_check_layout(self._h, _ptr(errs), ctypes.byref(info), _stream()), "pdp_debug_check_layout")
        return errs.cpu().tolist(), dict(blocked=int(info[0]) & 15, ctas=int(info[0]) >> 4, nvb=int(info[1]), ncb=int(info[2]), sv=int(info[3]), sc=int(info[4]))

    def check_edge_mask(self):
        """[variable-side, clause-side] counts of edge-mask bits that disagree with the node masks (tests)"""
        errs = self._new(2, dtype=torch.int32)
        self._check(self._L.pdp_debug_check_edge_mask(self._h, _ptr(errs), _stream()), "pdp_debug_check_edge_mask")
        return errs.cpu().tolist()

    def launch_count(self):
        return int(self._L.pdp_launch_count(self._h))

    # ---- stateless operators -----------------------------------------------------------------
    def cnf_eval(self, prediction):
        pred = _f32(prediction, self.device).reshape(-1)
        solved, nun = self._new(self.B), self._new(self.B)
        self._check(self._L.pdp_cnf_eval(self._h, _ptr(pred), _ptr(solved), _ptr(nun), _stream()), "pdp_cnf_eval")
        return solved, nun

    def energy(self, assignment, av, af):
        a, v, f = (_f32(x, self.device).reshape(-1) for x in (assignment, av, af))
        en, uf = self._new(self.B), self._new(self.F)
        self._check(self._L.pdp_energy(self._h, _ptr(a), _ptr(v), _ptr(f), _ptr(en), _ptr(uf), _stream()), "pdp_energy")
        return en, uf

    def energy_diff(self, assignment, av, edge_mask):
        a, v, em = (_f32(x, self.device).reshape(-1) for x in (assignment, av, edge_mask))
        d = self._new(self.V)
        self._check(self._L.pdp_energy_diff(self._h, _ptr(a), _ptr(v), _ptr(em), _ptr(d), _stream()), "pdp_energy_diff")
        return d

    def sp_step(self, dec_q3, dec_fs2, edge_mask=None, prop_q3=None, prop_fs2=None, active=None, pi=0.0):
        dq, df = _f32(dec_q3, self.device), _f32(dec_fs2, self.device)
        pq, pf = _f32(prop_q3, self.device), _f32(prop_fs2, self.device)
        em = None if edge_mask is None else _f32(edge_mask, self.device).reshape(-1)
        act = None if active is None else active.to(device=self.device, dtype=torch.uint8).reshape(-1).contiguous()
        oq, of = self._new(self.E, 3), self._new(self.E, 2)
        self._check(self._L.pdp_sp_step(self._h, _ptr(dq), _ptr(df), _ptr(em), _ptr(pq), _ptr(pf), _ptr(act), float(pi),
                                  _ptr(oq), _ptr(of), _stream()), "pdp_sp_step")
        return oq, of

    def sp_step_adapted(self, x_log, eta_in, ext_in, edge_mask, prop_q3, prop_fs2, active=None, pi=0.0):
        x, e, t = (_f32(v, self.device).reshape(-1) for v in (x_log, eta_in, ext_in))
        pq, pf = _f32(prop_q3, self.device), _f32(prop_fs2, self.device)
        em = None if edge_mask is None else _f32(edge_mask, self.device).reshape(-1)
        act = None if active is None else active.to(device=self.device, dtype=torch.uint8).reshape(-1).contiguous()
        oq, of = self._new(self.E, 3), self._new(self.E, 2)
        self._check(self._L.pdp_sp_step_adapted(self._h, _ptr(x), _ptr(e), _ptr(t), _ptr(em), _ptr(pq), _ptr(pf), _ptr(act), float(pi),
                                                _ptr(oq), _ptr(of), _stream()), "pdp_sp_step_adapted")
        return oq, of

    def edge_aggregate(self, state, by_variable=True, leave_one_out=False):
        """(node_sum [V|F, C], edge_loo [E, C] or None) of an [E, C] edge tensor (MessageAggregator's segmented sums)"""
        st = _f32(state, self.device)
        C = int(st.shape[1])
        out = self._new(self.V if by_variable else self.F, C)
        loo = self._new(self.E, C) if leave_one_out else None
        self._check(self._L.pdp_edge_aggregate(self._h, 1 if by_variable else 0, _ptr(st), C, _ptr(out), _ptr(loo), _stream()),
                    "pdp_edge_aggregate")
        return out, loo

    def score(self, fs2, af, pi=0.0):
        f, a = _f32(fs2, self.device), _f32(af, self.device).reshape(-1)
        s = self._new(self.V)
        self._check(self._L.pdp_score(self._h, _ptr(f), _ptr(a), float(pi), _ptr(s), _stream()), "pdp_score")
        return s

    # ---- solver state --------------------------------------------------------------------------
    def load_state(self, prop_state, dec_state):
        pq, pf = _f32(prop_state[0], self.device), _f32(prop_state[1], self.device)
        dq, df = _f32(dec_state[0], self.device), _f32(dec_state[1], self.device)
        self._check(self._L.pdp_load_state(self._h, _ptr(pq), _ptr(pf), _ptr(dq), _ptr(df), _stream()), "pdp_load_state")

    def load_state_const(self, qu, qs, qd, eta, ext):
        self._check(self._L.pdp_load_state_const(self._h, float(qu), float(qs), float(qd), float(eta), float(ext), _stream()),
                    "pdp_load_state_const")

    def store_state(self):
        q, f = self._new(self.E, 3), self._new(self.E, 2)
        self._check(self._L.pdp_store_state(self._h, _ptr(q), _ptr(f), _stream()), "pdp_store_state")
        return q, f

    def set_masks(self, av=None, af=None, solution=None):
        a = None if av is None else _f32(av, self.device).reshape(-1)
        f = None if af is None else _f32(af, self.device).reshape(-1)
        s = None if solution is None else _f32(solution, self.device).reshape(-1)
        self._check(self._L.pdp_set_masks(self._h, _ptr(a), _ptr(f), _ptr(s), _stream()), "pdp_set_masks")

    def set_active(self, active):
        a = active.to(device=self.device, dtype=torch.uint8).reshape(-1).contiguous()
        self._check(self._L.pdp_set_active(self._h, _ptr(a), _stream()), "pdp_set_active")

    def get_masks(self, edge_mask=False):
        av, af, sol = self._new(self.V), self._new(self.F), self._new(self.V)
        is_sat = self._new(self.B)
        active = self._new(self.B, dtype=torch.uint8)
        em = self._new(self.E) if edge_mask else None
        self._check(self._L.pdp_get_masks(self._h, _ptr(av), _ptr(af), _ptr(sol), _ptr(is_sat), _ptr(active), _ptr(em),
                                    _stream()), "pdp_get_masks")
        return dict(av=av, af=af, sol=sol, is_sat=is_sat, active=active, em=em)

    def solution(self):
        sol = self._new(self.V)
        self._check(self._L.pdp_get_masks(self._h, None, None, _ptr(sol), None, None, None, _stream()), "pdp_get_masks")
        return sol

    def problem_flags(self):
        flags = self._new(self.B, dtype=torch.int32)
        counters = self._new(self.B, dtype=torch.int32)
        freeze = self._new(self.B, dtype=torch.int32)
        self._check(self._L.pdp_get_problem_flags(self._h, _ptr(flags), _ptr(counters), _ptr(freeze), _stream()),
              "pdp_get_problem_flags")
        return flags, counters, freeze

    def simplify(self):
        self._check(self._L.pdp_simplify(self._h, _stream()), "pdp_simplify")

    def set_variables(self, assignment):
        a = _f32(assignment, self.device).reshape(-1)
        self._check(self._L.pdp_set_variables(self._h, _ptr(a), _stream()), "pdp_set_variables")

    def set_decimation_fraction(self, fraction):
        """SP-inspired decimation in sp_run: every selected problem fixes max(1, floor(fraction * active variables)) of its
        most biased variables per decimation step; 0 (the default) is the reference's one arg-max variable.  The value
        stays until the next call (pdp_reset keeps it)."""
        self._check(self._L.pdp_set_decimation_fraction(self._h, float(fraction)), "pdp_set_decimation_fraction")

    def decimation_select(self, coeff, score, fraction, problem_sel=None):
        """The decimation rule (arg-max for K_b == 1, top-K_b otherwise) on given coefficients [V] (>= 0) and scores [V]:
        returns the assignment [V] with sign(score) on the taken variables and 0 elsewhere.  problem_sel [B] (nonzero =
        converged and active; None = every problem); K_b counts the context's active variables."""
        c, sc = _f32(coeff, self.device).reshape(-1), _f32(score, self.device).reshape(-1)
        ps = None if problem_sel is None else problem_sel.to(device=self.device, dtype=torch.uint8).reshape(-1).contiguous()
        out = self._new(self.V)
        self._check(self._L.pdp_decimation_select(self._h, _ptr(c), _ptr(sc), _ptr(ps), float(fraction), _ptr(out), _stream()),
                    "pdp_decimation_select")
        return out

    def enable_conflict_rollback(self, on=True):
        """Conflict rollback for SP-inspired decimation in sp_run (include/pdp_b200.h, pdp_set_conflict_rollback): a step of
        K_b >= 2 variables that ends in a unit-propagation conflict is undone and the problem's later steps are halved.  The
        context allocates the snapshot buffer; on=False turns rollback off and frees it.  pdp_reset keeps the setting."""
        if not on:
            self._check(self._L.pdp_set_conflict_rollback(self._h, None, 0), "pdp_set_conflict_rollback")
            self._rb_scratch = None
            return
        nbytes = int(self._L.pdp_rollback_scratch_bytes(self.V, self.F, self.B))
        scratch = self._new(max(nbytes, 1), dtype=torch.uint8)
        self._check(self._L.pdp_set_conflict_rollback(self._h, _ptr(scratch), nbytes), "pdp_set_conflict_rollback")
        self._rb_scratch = scratch

    def set_reinforce(self, coins, decimation_probability=0.5):
        """Model type `reinforce` in sp_run (include/pdp_b200.h, pdp_set_reinforce): iteration k of the runs from here on
        draws coins[k] (fp32 [n] on the device) and, when it is < decimation_probability, sets every active problem's
        external forces to the signs of its SP biases; the retire test and the predictor replace the decimation.  coins=None
        turns the mode off.  The context keeps a reference to the coins while the mode is on."""
        if coins is None:
            self._check(self._L.pdp_set_reinforce(self._h, None, 0, 0.0), "pdp_set_reinforce")
            self._rf_coins = None
            return
        c = _f32(coins, self.device).reshape(-1).contiguous()
        self._check(self._L.pdp_set_reinforce(self._h, _ptr(c), int(c.numel()), float(decimation_probability)),
                    "pdp_set_reinforce")
        self._rf_coins = c

    def rollbacks(self):
        """(count int32 [B], iteration of the last rollback int32 [B], 0 = none) since pdp_reset"""
        count, last = self._new(self.B, dtype=torch.int32), self._new(self.B, dtype=torch.int32)
        self._check(self._L.pdp_get_rollbacks(self._h, _ptr(count), _ptr(last), _stream()), "pdp_get_rollbacks")
        return count, last

    def enable_trace(self, capacity=1 << 16):
        self._trace = torch.zeros(capacity, 3, dtype=torch.int32, device=self.device)
        self._check(self._L.pdp_set_trace_buffer(self._h, _ptr(self._trace), capacity), "pdp_set_trace_buffer")

    def disable_trace(self):
        self._check(self._L.pdp_set_trace_buffer(self._h, None, 0), "pdp_set_trace_buffer")
        self._trace = None

    def trace(self):
        n = ctypes.c_int32(0)
        self._check(self._L.pdp_trace_length(self._h, ctypes.byref(n), _stream()), "pdp_trace_length")
        return self._trace[: n.value].cpu()

    def sp_run(self, iterations, tolerance, t_max, check_termination=True, batch_replication=1, pi=0.0,
               full_state=False, sync=False, generic=False, grid_decimation=False, full_closure=False,
               caller_terminates=False):
        """T iterations of propagate/decimate/predict in one persistent kernel.  Returns the device
        int32 tensor holding the number of executed iterations (or the int when sync=True).
        generic=True forces the thread-per-node passes (A/B against the blocked shared-memory passes);
        grid_decimation=True the grid-wide decimation phases; full_closure=True their full-scan UP / peel closure."""
        prm = SpParams(int(iterations), float(tolerance), int(t_max), float(pi), 1 if check_termination else 0,
                       int(batch_replication), 1 if full_state else 0, (1 if generic else 0) | (2 if grid_decimation else 0) | (4 if full_closure else 0) | (8 if caller_terminates else 0) | int(os.environ.get("PDP_B200_SP_FLAGS", "0"), 0))
        self._timed("sp_run", lambda: self._check(
            self._L.pdp_sp_run(self._h, ctypes.byref(prm), _ptr(self._iters), _stream()), "pdp_sp_run"))
        if sync:
            return int(self._iters[0].item())
        return self._iters[:1]

    def count_active_variables(self):
        n = ctypes.c_int64(0)
        self._check(self._L.pdp_count_active_variables(self._h, ctypes.byref(n), _stream()), "pdp_count_active_variables")
        return int(n.value)

    def random_fill(self, draws):
        d = _f32(draws, self.device).reshape(-1)
        self._check(self._L.pdp_random_fill(self._h, _ptr(d), _stream()), "pdp_random_fill")

    def walksat(self, iterations, epsilon, rand_var=None, rand_coin=None, seed=0, batch_replication=1, sync=False):
        rv = None if rand_var is None else _f32(rand_var, self.device).reshape(-1)
        rc = None if rand_coin is None else _f32(rand_coin, self.device).reshape(-1)
        pred = self._new(self.V)
        self._timed("walksat", lambda: self._check(
            self._L.pdp_walksat(self._h, int(iterations), float(epsilon), int(batch_replication), _ptr(rv), _ptr(rc),
                                int(seed) & 0xFFFFFFFFFFFFFFFF, _ptr(pred), _ptr(self._iters[1:]), _stream()),
            "pdp_walksat"))
        if sync:
            return pred, int(self._iters[1].item())
        return pred, self._iters[1:]

    def deduplicate(self, batch_replication, prediction):
        p = _f32(prediction, self.device).reshape(-1)
        out = self._new(self.V // batch_replication)
        win = self._new(self.B // batch_replication, dtype=torch.int32)
        self._check(self._L.pdp_deduplicate(self._h, int(batch_replication), _ptr(p), _ptr(out), _ptr(win), _stream()),
              "pdp_deduplicate")
        return out, win
