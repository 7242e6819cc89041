"""Decimators of the PDP framework, B200-native (reference src/pdp/nn/pdp_decimate.py)."""
import math

import torch
import torch.nn as nn

from . import tensor_ops
from .pdp_propagate import edge_problem_mask


def smooth_max_by_variable(ctx, x):
    """sparse_smooth_max over each variable's edges (reference util.py:282-286, alpha = 30):
    sum(x * e^min(30x,30)) / max(sum(e^min(30x,30)), 1), sums by the library's segmented-sum kernel in ascending
    edge order"""
    w = torch.exp(torch.clamp(30.0 * x, max=30.0))
    s, _ = ctx.edge_aggregate(torch.stack((x * w, w), 1), by_variable=True)
    return s[:, 0] / torch.clamp(s[:, 1], min=1.0)


def problem_max(x, bvm, B):
    """sparse_max (reference util.py:267-275) with its rounding fl(fl(max fl(fl(x - min) + 1) + min) - 1) and its
    zero floor, `min` taken per problem (every problem behaves as in a batch of one, DESIGN.md section 4)"""
    idx = bvm.long()
    mn = torch.full((B,), float("inf"), dtype=x.dtype, device=x.device).scatter_reduce(0, idx, x, "amin", include_self=True)
    y = (x - mn[idx]) + 1.0
    mx = torch.zeros(B, dtype=x.dtype, device=x.device).scatter_reduce(0, idx, y, "amax", include_self=True)
    return (mx + mn) - 1.0


def problem_argmax(x, bvm, B):
    "sparse_argmax (reference util.py:257-265): first index of the per-problem maximum of fl(fl(x - min) + 1)"
    idx = bvm.long()
    V = x.shape[0]
    mn = torch.full((B,), float("inf"), dtype=x.dtype, device=x.device).scatter_reduce(0, idx, x, "amin", include_self=True)
    y = (x - mn[idx]) + 1.0
    mx = torch.zeros(B, dtype=x.dtype, device=x.device).scatter_reduce(0, idx, y, "amax", include_self=True)
    pos = torch.where(y == mx[idx], torch.arange(V, device=x.device), torch.full((1,), V, device=x.device))
    return torch.full((B,), V, dtype=torch.int64, device=x.device).scatter_reduce(0, idx, pos, "amin", include_self=True)


def check_decimation_fraction(fraction):
    """the fraction of SP-inspired decimation: a finite float with 0 <= f < 1 (0 = one arg-max variable per step)"""
    try:
        f = float(fraction)
    except (TypeError, ValueError):
        raise ValueError("decimation_fraction must be a number, got %r" % (fraction,))
    if not math.isfinite(f) or not 0.0 <= f < 1.0:
        raise ValueError("decimation_fraction must be finite with 0 <= f < 1, got %r" % (fraction,))
    return f


def check_conflict_rollback(conflict_rollback, fraction):
    """conflict rollback of SP-inspired decimation: a bool, and True only with a decimation fraction > 0"""
    if not isinstance(conflict_rollback, bool):
        raise ValueError("conflict_rollback must be True or False, got %r" % (conflict_rollback,))
    if conflict_rollback and fraction == 0.0:
        raise ValueError("conflict_rollback needs a decimation_fraction > 0 (one variable per step is never rolled back)")
    return conflict_rollback


def draw_coins(T, device):
    """The coins of T reinforce iterations drawn before a fused run: T separate torch.rand(1) draws on `device`, the values
    the step loop draws one per iteration (ReinforceDecimator._coin).  Returns (coins [T], the generator state before the
    draws) for settle_coins."""
    device = torch.device(device)
    state = torch.cuda.get_rng_state(device) if device.type == "cuda" else torch.get_rng_state()
    coins = torch.empty(int(T), dtype=torch.float32, device=device)
    for t in range(int(T)):
        torch.rand(1, out=coins[t:t + 1])
    return coins, state


def settle_coins(state, done, device):
    """Leaves the generator of `device` where a step loop that ran `done` iterations leaves it: back to `state` (from
    draw_coins), then `done` single draws again.  The draws that follow the run (WalkSAT) are then the step loop's."""
    device = torch.device(device)
    if device.type == "cuda":
        torch.cuda.set_rng_state(state, device)
    else:
        torch.set_rng_state(state)
    for _ in range(int(done)):
        torch.rand(1, device=device)


class NeuralDecimator(nn.Module):
    """The neural (non-greedy) decimator of `p-nd-np` / `np-nd-np` (reference pdp_decimate.py:21-100): one GRU
    cell per message direction over the edges; same sub-module names (state-dict compatible).  The GRU cells run on the
    tensor cores (pdp_edge_gru_forward: tcgen05 tf32 three-term split = fp32 accuracy, gates fused); PDP_B200_NN=torch
    keeps them on the library GEMMs for A/B comparisons.

    message_dimension == (3, 1) is widened to (3, 2) as the reference needs to run at all: its SurveyPropagator
    returns a 2-column function state (pdp_propagate.py:221) while solver.py:555 sizes the cell for 1 (SURVEY.md
    section 5, bit-rot item 4)."""

    def __init__(self, device, message_dimension, meta_data_dimension, hidden_dimension, mem_hidden_dimension,
                 mem_agg_hidden_dimension, agg_hidden_dimension, edge_dimension, dropout):
        super(NeuralDecimator, self).__init__()
        self._device = device
        self._module_list = nn.ModuleList()
        self._drop_out = dropout
        if message_dimension == (3, 1):
            message_dimension = (3, 2)
        if isinstance(message_dimension, tuple):
            variable_message_dim, function_message_dim = message_dimension
        else:
            variable_message_dim = function_message_dim = message_dimension
        self._variable_rnn_cell = nn.GRUCell(variable_message_dim + edge_dimension + meta_data_dimension, hidden_dimension, bias=True)
        self._function_rnn_cell = nn.GRUCell(function_message_dim + edge_dimension + meta_data_dimension, hidden_dimension, bias=True)
        self._module_list.append(self._variable_rnn_cell)
        self._module_list.append(self._function_rnn_cell)
        self._hidden_dimension = hidden_dimension
        self._mem_hidden_dimension = mem_hidden_dimension
        self._agg_hidden_dimension = agg_hidden_dimension
        self._mem_agg_hidden_dimension = mem_agg_hidden_dimension

    def forward(self, init_state, message_state, sat_problem, is_training, active_mask=None):
        if sat_problem._meta_data is not None:
            raise NotImplementedError("meta_data features are not supported")
        mask = edge_problem_mask(sat_problem, active_mask)
        variable_state, function_state = message_state[0], message_state[1]
        ef = sat_problem._edge_feature
        if tensor_ops.use_tensor_cores():
            # both GRU cells on the tensor cores, gates and the frozen-problem blend fused in the epilogue (csrc/pdp_edge_nn.cu)
            tc = self.__dict__.setdefault("_tc_cells", {})
            if not tc:
                tc["v"] = tensor_ops.TensorGRU(self._variable_rnn_cell)
                tc["f"] = tensor_ops.TensorGRU(self._function_rnn_cell)
            return (tc["v"]([variable_state, ef], init_state[0], row_mask=mask),
                    tc["f"]([function_state, ef], init_state[1], row_mask=mask))
        new_v = self._variable_rnn_cell(torch.cat((variable_state, ef), 1), init_state[0])
        new_f = self._function_rnn_cell(torch.cat((function_state, ef), 1), init_state[1])
        if mask is not None:   # frozen problems keep their state (reference :75,83)
            new_v = mask * new_v + (1 - mask) * init_state[0]
            new_f = mask * new_f + (1 - mask) * init_state[1]
        return new_v, new_f

    def get_init_state(self, graph_map, batch_variable_map, batch_function_map, edge_feature, graph_feat,
                       randomized, batch_replication):
        "reference pdp_decimate.py:89-100"
        edge_num = graph_map.size(1) * batch_replication
        if randomized:
            variable_state = 2.0 * torch.rand(edge_num, self._hidden_dimension, dtype=torch.float32, device=self._device) - 1.0
            function_state = 2.0 * torch.rand(edge_num, self._hidden_dimension, dtype=torch.float32, device=self._device) - 1.0
        else:
            variable_state = torch.zeros(edge_num, self._hidden_dimension, dtype=torch.float32, device=self._device)
            function_state = torch.zeros(edge_num, self._hidden_dimension, dtype=torch.float32, device=self._device)
        return (variable_state, function_state)


class SequentialDecimator(nn.Module):
    """The greedy, convergence-gated sequential decimator (reference pdp_decimate.py:106-183): at most
    one variable per problem and iteration is fixed, once that problem's surveys have converged
    (max smooth-max |delta eta| < tolerance) or its counter reached t_max.

    decimation_fraction f > 0 turns it into SP-inspired decimation: a selected problem with A active variables fixes
    the max(1, floor(f * A)) variables with the largest |score| at once (include/pdp_b200.h, pdp_decimation_select).
    conflict_rollback (needs f > 0) undoes a step of two or more variables that ends in a unit-propagation conflict and
    halves the problem's later steps (pdp_set_conflict_rollback).  Both are plain attributes, not buffers: state dicts of
    the reference load unchanged.

    Its statistics, per-problem decisions, scoring, arg-max, variable fixing and the following unit
    propagation / peeling closure all live inside the persistent kernel launched by
    PropagatorDecimatorSolverBase.forward (pdp_sp_run); the module keeps the hyper-parameters and the
    initial-state contract."""

    def __init__(self, device, message_dimension, scorer, tolerance, t_max, decimation_fraction=0.0, conflict_rollback=False):
        super(SequentialDecimator, self).__init__()
        self._decimation_fraction = check_decimation_fraction(decimation_fraction)
        self._conflict_rollback = check_conflict_rollback(conflict_rollback, self._decimation_fraction)
        self._device = device
        self._tolerance = tolerance
        self._scorer = scorer
        self._message_dimension = message_dimension
        self._t_max = t_max
        self._previous_function_state = None
        self._counters = None
        self.decimation_log = []          # (variable indices, signs) of every stepwise decimation (diagnostics, tests)
        self._module_list = nn.ModuleList([self._scorer])

    def forward(self, init_state, message_state, sat_problem, is_training, active_mask=None):
        """One decimation step on the library's stateless operators (reference pdp_decimate.py:122-177), for
        scorers other than the SurveyScorer (model type np-d-np); p-d-p never comes here, its decimator runs inside
        the persistent kernel."""
        ctx = sat_problem._ctx
        B, V, bvm = ctx.B, ctx.V, sat_problem._batch_variable_map
        idx = bvm.long()
        if self._counters is None:
            self._counters = torch.zeros(B, device=ctx.device)
        av = ctx.get_masks()["av"]
        eta = message_state[1][:, 0]
        if active_mask is not None:
            survey = problem_max(smooth_max_by_variable(ctx, eta) * av, bvm, B)
            active_mask[survey <= 1e-10, 0] = 0
        if self._previous_function_state is not None and bool((av.sum() > 0).item()):
            diff = (self._previous_function_state - eta).abs()
            em = sat_problem._edge_mask
            if em is not None:
                diff = diff * em[:, 0]
            sum_diff = problem_max(smooth_max_by_variable(ctx, diff) * av, bvm, B)
            self._counters[sum_diff < self._tolerance] = 0
            conv = (sum_diff < self._tolerance).float()
            conv[self._counters >= self._t_max] = 1
            self._counters[self._counters >= self._t_max] = 0
            conv_v = conv[idx]
            if bool((conv_v.sum() > 0).item()):
                score = self._scorer(message_state, sat_problem)[0][:, 0]
                coeff = score.abs() * av * conv_v
                if bool((coeff.sum() > 0).item()) and self._decimation_fraction > 0.0:
                    sel = None if active_mask is None else active_mask[:, 0]
                    assignment = ctx.decimation_select(coeff, score, self._decimation_fraction, sel)
                    ind = torch.nonzero(assignment).reshape(-1)
                    if ind.numel() > 0:
                        sat_problem.set_variables(assignment)
                        self.decimation_log.append((ind, assignment[ind].clone()))
                elif bool((coeff.sum() > 0).item()):
                    max_ind = problem_argmax(coeff, bvm, B)
                    norm = torch.zeros(B, device=ctx.device).index_add_(0, idx, coeff)
                    sel = norm != 0
                    if active_mask is not None:
                        sel = sel & (active_mask[:, 0] != 0)
                    max_ind = max_ind[sel]
                    if max_ind.numel() > 0:
                        assignment = torch.zeros(V, device=ctx.device)
                        assignment[max_ind] = score.sign()[max_ind]
                        sat_problem.set_variables(assignment)
                        self.decimation_log.append((max_ind.clone(), assignment[max_ind].clone()))
            self._counters = self._counters + 1
        self._previous_function_state = eta
        return message_state

    def get_init_state(self, graph_map, batch_variable_map, batch_function_map, edge_feature, graph_feat,
                       randomized, batch_replication):
        "reference pdp_decimate.py:179-183: module state is reset, the scorer provides the messages"
        self._previous_function_state = None
        self._counters = None
        self.decimation_log = []
        return self._scorer.get_init_state(graph_map, batch_variable_map, batch_function_map, edge_feature,
                                           graph_feat, randomized, batch_replication)


class ReinforceDecimator(nn.Module):
    """The (distributed) Reinforce decimator of model type `reinforce` (reference pdp_decimate.py:189-250): no variable
    is fixed; with probability `decimation_probability` per iteration (one batch-global coin, pdp_decimate.py:218)
    every edge's external force becomes the sign of its variable's SP bias, which the propagator and scorer feed
    back through their pi terms.  Problems whose surveys moved by at most 0.01 are retired.

    Inside ReinforceSurveyPropagatorSolver.forward the whole loop runs in the persistent kernel (pdp_set_reinforce) with
    coins drawn beforehand (draw_coins / settle_coins), unless `_coin_source` is set or the caller's termination callback
    is its own: then forward() below runs once per iteration."""

    _draws_per_iteration = True       # one coin per iteration: the solver loop must stop exactly where the reference stops

    def __init__(self, device, scorer, decimation_probability=0.5):
        super(ReinforceDecimator, self).__init__()
        self._device = device
        self._scorer = scorer
        self._decimation_probability = decimation_probability
        self._function_message_dim = 3
        self._variable_message_dim = 2
        self._previous_function_state = None
        self._coin_source = None          # tests: callable returning the next coin instead of torch.rand

    def _coin(self):
        if self._coin_source is not None:
            return float(self._coin_source())
        return float(torch.rand(1, device=self._device).item())

    def forward(self, init_state, message_state, sat_problem, is_training, active_mask=None):
        ctx = sat_problem._ctx
        variable_state, function_state = message_state[0], message_state[1]
        eta = function_state[:, 0]
        if active_mask is not None and self._previous_function_state is not None:
            av = ctx.get_masks()["av"]
            if bool((av.sum() > 0).item()):
                diff = (self._previous_function_state - eta).abs()
                em = sat_problem._edge_mask
                if em is not None:
                    diff = diff * em[:, 0]
                sum_diff = problem_max(smooth_max_by_variable(ctx, diff) * av, sat_problem._batch_variable_map, ctx.B)
                active_mask[sum_diff <= 0.01, 0] = 0
        self._previous_function_state = eta.clone()
        if self._coin() < self._decimation_probability:
            score = self._scorer(message_state, sat_problem)[0][:, 0]
            force = torch.sign(score)[sat_problem._graph_map[0].long()]
            mask = edge_problem_mask(sat_problem, active_mask)
            if mask is None:
                function_state[:, 1] = force
            else:
                m = mask[:, 0]
                function_state[:, 1] = m * force + (1 - m) * function_state[:, 1]
        return variable_state, function_state

    def get_init_state(self, graph_map, batch_variable_map, batch_function_map, edge_feature, graph_feat,
                       randomized, batch_replication):
        "reference pdp_decimate.py:236-250"
        self._previous_function_state = None
        edge_num = graph_map.size(1) * batch_replication
        if randomized:
            variable_state = torch.rand(edge_num, self._function_message_dim, dtype=torch.float32, device=self._device)
            function_state = torch.rand(edge_num, self._variable_message_dim, dtype=torch.float32, device=self._device)
        else:
            variable_state = torch.ones(edge_num, self._function_message_dim, dtype=torch.float32,
                                        device=self._device) / self._function_message_dim
            function_state = 0.5 * torch.ones(edge_num, self._variable_message_dim, dtype=torch.float32, device=self._device)
        function_state[:, 1] = 0
        return (variable_state, function_state)
