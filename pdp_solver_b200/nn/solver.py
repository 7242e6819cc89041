"""Drop-in for the reference module `pdp.nn.solver` (reference src/pdp/nn/solver.py), B200-native.

Same class names, constructor arguments, `get_init_state` / `forward` signatures and return layout as
the reference; underneath, the batch lives in a device `Context` (CSR/CSC instead of 14 torch sparse
matrices) and the whole propagate -> decimate -> predict loop, the CNF check, unit propagation /
peeling and WalkSAT run as hand-written sm_100a kernels behind the C ABI of libpdp_b200.so.

Scope (SURVEY.md section 8): the classical model types `p-d-p` (SurveyPropagatorSolver), `walk-sat` (WalkSATSolver) and
`reinforce` (ReinforceSurveyPropagatorSolver) run entirely in the library's kernels (one persistent launch for the whole
loop).  The neural
model types `p-nd-np` (NeuralSurveyPropagatorSolver) and `np-nd-np` (NeuralPropagatorDecimatorSolver) run the
reference's iteration structure step by step: message arithmetic, segmented sums, CNF check, simplification and
WalkSAT are the library's kernels, the dense layers (Linear adaptors, GRU cells, MLPs) are library GEMMs through
torch in fp32.  There is no CPU path and no fallback: CPU tensors or a missing library raise.
"""
import os
import warnings

import torch
import torch.nn as nn

from .. import _lib
from ..engine import Context
from . import pdp_decimate, pdp_predict, pdp_propagate, util

# WalkSAT draws are pre-generated with torch.rand in the reference's order when they fit this many
# floats; above it the kernel's counter-based generator is used (same distribution, other stream).
TORCH_RNG_DRAW_LIMIT = int(os.environ.get("PDP_TORCH_RNG_DRAW_LIMIT", str(1 << 24)))


class SATProblem(object):
    """One batch of CNFs on the device (reference solver.py:19-285).  Exposes the attributes the
    reference's callbacks read (`_graph_map`, `_batch_variable_map`, `_batch_function_map`,
    `_edge_feature`, `_meta_data`, `_batch_replication`, `_active_variables`, `_active_functions`,
    `_solution`, `_edge_mask`, `_batch_size`, ...); the mask attributes are fetched from the device
    context on access."""

    def __init__(self, data_batch, device, batch_replication=1):
        self._device = device
        self._batch_replication = batch_replication
        graph_map, bvm, bfm, edge_feature, meta_data, _ = data_batch
        if graph_map.device.type != "cuda":
            raise _lib.PdpError("pdp_solver_b200 runs on CUDA tensors only (there is no CPU path); "
                                "move the batch to the GPU as the reference's _to_cuda does")
        self._replication_mask_tuple = None
        if batch_replication > 1:
            graph_map, bvm, bfm, edge_feature, meta_data = self._replicate_batch(
                graph_map, bvm, bfm, edge_feature, meta_data, batch_replication)
        self._graph_map, self._batch_variable_map, self._batch_function_map = graph_map, bvm, bfm
        self._edge_feature, self._meta_data = edge_feature, meta_data
        self._variable_num = bvm.size(0)
        self._function_num = bfm.size(0)
        self._edge_num = graph_map.size(1)
        self._ctx = Context(graph_map, bvm, bfm, edge_feature)
        self._batch_size = self._ctx.B
        self._edge_mask_set = False
        if batch_replication > 1:
            self._replication_mask_tuple = self._compute_batch_replication_map(batch_replication)

    @staticmethod
    def _replicate_batch(graph_map, bvm, bfm, edge_feature, meta_data, b):
        """replica r of problem j gets problem id r*B + j (reference solver.py:56-82)"""
        V, F = bvm.size(0), bfm.size(0)
        B = int(bvm.max().item()) + 1
        r = torch.arange(b, dtype=torch.int32, device=graph_map.device)
        off = torch.stack([r * V, r * F])                                  # [2, b]
        gm = (graph_map.unsqueeze(1) + off.unsqueeze(2)).reshape(2, -1)    # [2, b*E]
        bv = (bvm.unsqueeze(0) + (r * B).unsqueeze(1)).reshape(-1)
        bf = (bfm.unsqueeze(0) + (r * B).unsqueeze(1)).reshape(-1)
        ef = edge_feature.repeat(b, 1)
        md = None if meta_data is None else meta_data.repeat(b, 1)
        return gm.contiguous(), bv.contiguous(), bf.contiguous(), ef, md

    def _compute_batch_replication_map(self, b):
        """dense-free equivalent of reference solver.py:84-99 for callbacks that torch.mm with it"""
        B0 = self._batch_size // b
        x = torch.arange(B0 * b, dtype=torch.int64, device=self._graph_map.device)
        ind = torch.stack([x, x % B0])
        with warnings.catch_warnings():
            warnings.simplefilter("ignore", UserWarning)     # "sparse invariant checks are implicitly disabled"
            mask = torch.sparse_coo_tensor(ind, torch.ones(B0 * b, device=self._graph_map.device), (B0 * b, B0))
        return (mask, mask.transpose(0, 1))

    def edge_problem_index(self):
        "problem id of every edge (int64 [E]), cached"
        if getattr(self, "_edge_problem", None) is None:
            self._edge_problem = self._batch_variable_map.long()[self._graph_map[0].long()]
        return self._edge_problem

    def update_solution(self, variable_prediction):
        """_update_solution (reference solver.py:388-399): active variables take the prediction, the others keep
        their solution; returns the merged [V,1] solution"""
        m = self._ctx.get_masks()
        av, sol = m["av"], m["sol"]
        merged = av * variable_prediction.reshape(-1) + (1.0 - av) * sol
        self._ctx.set_masks(solution=torch.where(av == 1, merged, sol))
        return merged.unsqueeze(1)

    # ---- state views -----------------------------------------------------------------------------
    @property
    def _active_variables(self):
        return self._ctx.get_masks()["av"].unsqueeze(1)

    @property
    def _active_functions(self):
        return self._ctx.get_masks()["af"].unsqueeze(1)

    @property
    def _solution(self):
        return self._ctx.solution()

    @property
    def _is_sat(self):
        return self._ctx.get_masks()["is_sat"]

    @property
    def _edge_mask(self):
        if not self._edge_mask_set:
            return None
        return self._ctx.get_masks(edge_mask=True)["em"].unsqueeze(1)

    # ---- reference solver.py:275-285 ---------------------------------------------------------------
    def set_variables(self, assignment):
        self._ctx.set_variables(assignment)

    def simplify(self):
        self._ctx.simplify()


def _const_rows(t):
    """the row every edge shares when `t` is an unmodified constant state of get_init_state, else None"""
    tag = getattr(t, "_pdp_const", None)
    if tag is None or tag[1] != t._version:
        return None
    return tag[0]


class _DeferredState(object):
    """(variable_state [E,3], function_state [E,2]) of the solver context, materialised in the caller's edge
    order on first access (pdp_store_state).  Behaves like the tuple the reference returns."""

    def __init__(self, ctx):
        self._ctx, self._value = ctx, None

    def _get(self):
        if self._value is None:
            self._value = tuple(self._ctx.store_state())
            self._ctx = None
        return self._value

    def __iter__(self):
        return iter(self._get())

    def __getitem__(self, i):
        return self._get()[i]

    def __len__(self):
        return 2


def _is_standard_termination(cb):
    """Only a callable explicitly tagged `_pdp_standard_termination` -- the trainer's own
    `_check_recurrence_termination` (reference trainer.py:150-162) carries the tag on its function object, so an
    override in a subclass does not -- is evaluated inside the persistent kernel; any other callable is called after
    every iteration, as the reference does."""
    return cb is not None and bool(getattr(cb, "_pdp_standard_termination", False))


class PropagatorDecimatorSolverBase(nn.Module):
    "The base class for all PDP SAT solvers (reference solver.py:293-511)."

    def __init__(self, device, name, propagator, decimator, predictor, local_search_iterations=0, epsilon=0.05):
        super(PropagatorDecimatorSolverBase, self).__init__()
        self._device = device
        self._module_list = nn.ModuleList()
        self._propagator, self._decimator, self._predictor = propagator, decimator, predictor
        for m in (propagator, decimator, predictor):
            self._module_list.append(m)
        self._global_step = nn.Parameter(torch.tensor([0], dtype=torch.float, device=self._device), requires_grad=False)
        self._name = name
        self._local_search_iterations = local_search_iterations
        self._epsilon = epsilon
        self.last_problem = None          # SATProblem of the last forward (flags, diagnostics)
        self.last_iterations = None

    def parameter_count(self):
        return sum(p.numel() for p in self.parameters() if p.requires_grad)

    def save(self, export_path_base):
        torch.save(self.state_dict(), os.path.join(export_path_base, self._name))

    def load(self, import_path_base):
        self.load_state_dict(torch.load(os.path.join(import_path_base, self._name)))

    def get_init_state(self, graph_map, batch_variable_map, batch_function_map, edge_feature, graph_feat,
                       randomized, batch_replication=1):
        "Initializes the propagator and the decimator messages in each direction (reference solver.py:498-511)."
        p = None if self._propagator is None else self._propagator.get_init_state(
            graph_map, batch_variable_map, batch_function_map, edge_feature, graph_feat, randomized, batch_replication)
        d = None if self._decimator is None else self._decimator.get_init_state(
            graph_map, batch_variable_map, batch_function_map, edge_feature, graph_feat, randomized, batch_replication)
        return p, d

    # ------------------------------------------------------------------------------------------
    def forward(self, init_state, graph_map, batch_variable_map, batch_function_map, edge_feature,
                meta_data, is_training=True, iteration_num=1, check_termination=None, simplify=True,
                batch_replication=1):
        """reference solver.py:324-353.  Returns (prediction, (propagator_state, decimator_state)) with
        prediction = (variable_prediction [V,1] in [0,1], None)."""
        if is_training:
            raise NotImplementedError("training (is_training=True) is outside the accelerated path (SURVEY.md section 8)")
        init_propagator_state, init_decimator_state = init_state
        self.last_problem = None   # releases the previous batch's workspace before the new one is allocated
        sat_problem = SATProblem((graph_map, batch_variable_map, batch_function_map, edge_feature, meta_data, None),
                                 self._device, batch_replication)
        ctx = sat_problem._ctx
        self.last_problem = sat_problem
        if simplify:
            sat_problem.simplify()

        propagator_state = decimator_state = None
        if self._propagator is not None and self._decimator is not None:
            fused = check_termination is None or _is_standard_termination(check_termination)
            if isinstance(self._decimator, pdp_decimate.SequentialDecimator) and \
                    isinstance(self._decimator._scorer, pdp_predict.SurveyScorer):
                propagator_state, decimator_state = self._forward_core(
                    init_propagator_state, init_decimator_state, sat_problem, iteration_num, check_termination)
            elif isinstance(self._decimator, pdp_decimate.ReinforceDecimator) and fused and \
                    self._decimator._coin_source is None:
                propagator_state, decimator_state = self._forward_core_reinforce(
                    init_propagator_state, init_decimator_state, sat_problem, iteration_num, check_termination)
            else:
                propagator_state, decimator_state = self._forward_core_stepwise(
                    init_propagator_state, init_decimator_state, sat_problem, iteration_num, check_termination)

        # predictor, last call.  IdentityPredictor: random fill of the undecided variables (pdp_predict.py:121-126);
        # a neural predictor's output becomes the solution of the active variables (solver.py:342,348)
        last = self._predictor(decimator_state, sat_problem, True)
        if not isinstance(self._predictor, pdp_predict.IdentityPredictor) and last[0] is not None:
            sat_problem.update_solution(last[0])
        prediction = self._local_search(sat_problem, batch_replication)
        if batch_replication > 1:
            prediction, winner = ctx.deduplicate(batch_replication, prediction)
            # states of the winning replicas (reference solver.py:417-424)
            if propagator_state is not None:
                propagator_state = decimator_state = self._dedup_states(propagator_state, sat_problem,
                                                                        batch_replication, winner)
        return (prediction.unsqueeze(1), None), (propagator_state, decimator_state)

    @staticmethod
    def _dedup_states(state, sat_problem, b, winner):
        E0 = sat_problem._edge_num // b
        gm = sat_problem._graph_map[:, :E0]
        prob = sat_problem._batch_variable_map[gm[0].long()].long()       # original problem of each edge
        src = winner.long()[prob] * E0 + torch.arange(E0, device=gm.device)
        return tuple(x[src] for x in state[:2])

    def _forward_core(self, init_propagator_state, init_decimator_state, sat_problem, iteration_num, check_termination):
        """reference solver.py:355-386 for the p-d-p composition: one persistent kernel when the
        termination callback is the trainer's (or None), one launch per iteration otherwise."""
        ctx = sat_problem._ctx
        dec = self._decimator
        if os.environ.get("PDP_PHASE_TIMING"):
            ctx.enable_trace(256)
        cq = _const_rows(init_decimator_state[0])
        cf = _const_rows(init_decimator_state[1])
        if cq is not None and cf is not None:
            ctx.load_state_const(cq[0], cq[1], cq[2], cf[0], cf[1])
        else:
            ctx.load_state(init_propagator_state, init_decimator_state[:2])
        b = sat_problem._batch_replication
        ctx.set_decimation_fraction(dec._decimation_fraction)
        if dec._conflict_rollback:
            ctx.enable_conflict_rollback()
        if check_termination is None or _is_standard_termination(check_termination):
            self.last_iterations = ctx.sp_run(iteration_num, dec._tolerance, dec._t_max,
                                              check_termination is not None, b, self._propagator.pi_value())
        else:
            # an arbitrary callback (reference solver.py:376-384): one iteration per launch, the callback sees the
            # active mask and the current solution and its verdict goes back into the context
            done = 0
            for _ in range(int(iteration_num)):
                if int(ctx.sp_run(1, dec._tolerance, dec._t_max, True, b, self._propagator.pi_value(), sync=True,
                                  caller_terminates=True)) == 0:
                    break
                done += 1
                m = ctx.get_masks()
                active_mask = m["active"].unsqueeze(1)
                check_termination(active_mask, (m["sol"].unsqueeze(1), None), sat_problem)
                ctx.set_active(active_mask[:, 0])
                if int(active_mask.sum().item()) <= 0:
                    break
            self.last_iterations = torch.tensor([done], dtype=torch.int32, device=ctx.device)
        sat_problem._edge_mask_set = iteration_num > 0
        # the final message states are exported on first use (the predict path never looks at them)
        state = _DeferredState(ctx)
        return state, state

    def _forward_core_reinforce(self, init_propagator_state, init_decimator_state, sat_problem, iteration_num,
                                check_termination):
        """reference solver.py:355-386 for model type `reinforce` in one persistent kernel (pdp_set_reinforce): the coins
        of all T iterations are drawn before the launch, and the generator is left where the step loop leaves it."""
        ctx = sat_problem._ctx
        dec = self._decimator
        ctx.load_state(init_propagator_state, init_decimator_state[:2])
        T = int(iteration_num)
        coins, rng_state = pdp_decimate.draw_coins(T, ctx.device)
        ctx.set_reinforce(coins, dec._decimation_probability)
        try:
            # the blocked passes where the batch allows; the returned [E,3] state is re-derived on export with the forces the
            # last sweep read (pdp_set_reinforce)
            done = ctx.sp_run(T, 0.0, 0, check_termination is not None, sat_problem._batch_replication,
                              self._propagator.pi_value(), sync=True)
        finally:
            ctx.set_reinforce(None)
        pdp_decimate.settle_coins(rng_state, done, ctx.device)
        self.last_iterations = torch.tensor([done], dtype=torch.int32, device=ctx.device)
        sat_problem._edge_mask_set = T > 0
        state = _DeferredState(ctx)
        return state, state

    def _forward_core_stepwise(self, init_propagator_state, init_decimator_state, sat_problem, iteration_num, check_termination):
        """reference solver.py:355-386 for the compositions that are not the fused p-d-p loop (p-nd-np, np-nd-np,
        np-d-np, reinforce), one iteration at a time like the reference.  Only the sequential decimator of np-d-np
        fixes variables; for the others the masks only change in the initial simplify()."""
        ctx = sat_problem._ctx
        propagator_state, decimator_state = init_propagator_state, init_decimator_state
        active_mask = None if check_termination is None else torch.ones(ctx.B, 1, dtype=torch.uint8, device=ctx.device)
        standard = check_termination is not None and _is_standard_termination(check_termination)
        rep = sat_problem._batch_replication
        fixes = isinstance(self._decimator, pdp_decimate.SequentialDecimator)
        # No host round trip inside the loop (the reference takes several per iteration, solver.py:365-384):
        #  * the edge mask always rides in the decimator state -- multiplying by an all-ones mask is exact, so whether
        #    anything is masked yet need not be known on the host;
        #  * the executed-iteration count lives on the device: an iteration counts iff some problem was active when it began;
        #  * "every problem has retired" reaches the host through a pinned flag copied asynchronously and looked at exactly
        #    two iterations later (deterministic: the same number of iterations -- and of random draws -- runs every time).
        #    The two iterations that run past that point change nothing: every message and hidden state of a retired
        #    problem is blended back (mask * new + (1 - mask) * old with mask 0), and the prediction is a function of
        #    those states.
        # (a decimator that draws random numbers every iteration -- reinforce -- and a caller's own termination callback
        #  keep the reference's immediate stop: extra iterations would consume draws / call the callback again)
        lag = 2 if (standard and not getattr(self._decimator, "_draws_per_iteration", False)) else 0
        edge_mask = ctx.get_masks(edge_mask=True)["em"].unsqueeze(1)
        done_dev = torch.zeros((), dtype=torch.int32, device=ctx.device)
        flags = torch.empty(2, dtype=torch.int32).pin_memory() if check_termination is not None else None
        events = [None, None]
        for it in range(int(iteration_num)):
            if flags is not None:
                ev = events[it & 1]
                if ev is not None:
                    ev.synchronize()       # (iteration it - 2: long finished unless the device is two iterations behind)
                    if int(flags[it & 1]) <= 0:
                        break
                done_dev += (active_mask.sum() > 0).to(torch.int32)
            else:
                done_dev += 1
            propagator_state = self._propagator(propagator_state, decimator_state, sat_problem, False, active_mask)
            decimator_state = self._decimator(decimator_state, propagator_state, sat_problem, False, active_mask)
            sat_problem._edge_mask_set = True
            if fixes:
                edge_mask = ctx.get_masks(edge_mask=True)["em"].unsqueeze(1)
            decimator_state = tuple(decimator_state[:2]) + (edge_mask,)     # solver.py:373-374
            if check_termination is not None:
                prediction = self._predictor(decimator_state, sat_problem)
                solution = sat_problem.update_solution(prediction[0])
                if standard:   # trainer._check_recurrence_termination (trainer.py:150-162) on the library's CNF check
                    solved, _ = ctx.cnf_eval(solution)
                    ok = solved > 0.5
                    if rep > 1:  # a solved replica retires every replica of its problem
                        ok = ok.reshape(rep, -1).any(0).repeat(rep)
                    active_mask[(active_mask[:, 0] == 1) & ok, 0] = 0
                else:
                    check_termination(active_mask, (solution, prediction[1]), sat_problem)
                if lag == 0:
                    if int(active_mask.sum().item()) <= 0:
                        break
                else:
                    flags[it & 1:(it & 1) + 1].copy_(active_mask.sum().to(torch.int32).reshape(1), non_blocking=True)
                    ev = torch.cuda.Event()
                    ev.record()
                    events[it & 1] = ev
        self.last_iterations = done_dev.reshape(1)
        return propagator_state, decimator_state

    def _local_search(self, sat_problem, batch_replication):
        "WalkSAT post-processing + solution merge (reference solver.py:433-467, 388-399)."
        ctx = sat_problem._ctx
        W = int(self._local_search_iterations)
        V, B = ctx.V, ctx.B
        if W > 0 and W * (V + B) <= TORCH_RNG_DRAW_LIMIT:
            # the reference's draw order per iteration: rand([V,1]) then rand(B) (solver.py:457,460)
            rv = torch.empty(W, V, device=ctx.device)
            rc = torch.empty(W, B, device=ctx.device)
            for it in range(W):
                torch.rand(V, out=rv[it])
                torch.rand(B, out=rc[it])
            pred, _ = ctx.walksat(W, self._epsilon, rv, rc, 0, batch_replication)
        else:
            seed = int(torch.randint(0, 2 ** 62, (1,)).item()) if W > 0 else 0
            pred, _ = ctx.walksat(W, self._epsilon, None, None, seed, batch_replication)
        return pred


class SurveyPropagatorSolver(PropagatorDecimatorSolverBase):
    "The classical SP-guided decimation solver, model type `p-d-p` (reference solver.py:567-578)."

    def __init__(self, device, name, tolerance, t_max, local_search_iterations=0, epsilon=0.05, decimation_fraction=0.0,
                 conflict_rollback=False):
        super(SurveyPropagatorSolver, self).__init__(
            device=device, name=name,
            propagator=pdp_propagate.SurveyPropagator(device, decimator_dimension=1, include_adaptors=False),
            decimator=pdp_decimate.SequentialDecimator(
                device, message_dimension=(3, 1),
                scorer=pdp_predict.SurveyScorer(device, message_dimension=1, include_adaptors=False),
                tolerance=tolerance, t_max=t_max, decimation_fraction=decimation_fraction,
                conflict_rollback=conflict_rollback),
            predictor=pdp_predict.IdentityPredictor(device=device, random_fill=True),
            local_search_iterations=local_search_iterations, epsilon=epsilon)


class WalkSATSolver(PropagatorDecimatorSolverBase):
    "The classical Walk-SAT solver, model type `walk-sat` (reference solver.py:584-592)."

    def __init__(self, device, name, iteration_num, epsilon=0.05):
        super(WalkSATSolver, self).__init__(
            device=device, name=name, propagator=None, decimator=None,
            predictor=pdp_predict.IdentityPredictor(device=device, random_fill=True),
            local_search_iterations=iteration_num, epsilon=epsilon)


class NeuralPropagatorDecimatorSolver(PropagatorDecimatorSolverBase):
    "The fully neural PDP solver, model type `np-nd-np` (reference solver.py:517-537)."

    def __init__(self, device, name, edge_dimension, meta_data_dimension, propagator_dimension, decimator_dimension,
                 mem_hidden_dimension, agg_hidden_dimension, mem_agg_hidden_dimension, prediction_dimension,
                 variable_classifier=None, function_classifier=None, dropout=0, local_search_iterations=0, epsilon=0.05):
        super(NeuralPropagatorDecimatorSolver, self).__init__(
            device=device, name=name,
            propagator=pdp_propagate.NeuralMessagePasser(device, edge_dimension, decimator_dimension, meta_data_dimension,
                                                         propagator_dimension, mem_hidden_dimension, mem_agg_hidden_dimension,
                                                         agg_hidden_dimension, dropout),
            decimator=pdp_decimate.NeuralDecimator(device, propagator_dimension, meta_data_dimension, decimator_dimension,
                                                   mem_hidden_dimension, mem_agg_hidden_dimension, agg_hidden_dimension,
                                                   edge_dimension, dropout),
            predictor=pdp_predict.NeuralPredictor(device, decimator_dimension, prediction_dimension, edge_dimension,
                                                  meta_data_dimension, mem_hidden_dimension, agg_hidden_dimension,
                                                  mem_agg_hidden_dimension, variable_classifier, function_classifier),
            local_search_iterations=local_search_iterations, epsilon=epsilon)
        self.to(device)


class NeuralSurveyPropagatorSolver(PropagatorDecimatorSolverBase):
    "SP propagator with neural adaptors + neural decimator, model type `p-nd-np` (reference solver.py:543-561)."

    def __init__(self, device, name, edge_dimension, meta_data_dimension, decimator_dimension, mem_hidden_dimension,
                 agg_hidden_dimension, mem_agg_hidden_dimension, prediction_dimension, variable_classifier=None,
                 function_classifier=None, dropout=0, local_search_iterations=0, epsilon=0.05):
        super(NeuralSurveyPropagatorSolver, self).__init__(
            device=device, name=name,
            propagator=pdp_propagate.SurveyPropagator(device, decimator_dimension, include_adaptors=True),
            decimator=pdp_decimate.NeuralDecimator(device, (3, 1), meta_data_dimension, decimator_dimension,
                                                   mem_hidden_dimension, mem_agg_hidden_dimension, agg_hidden_dimension,
                                                   edge_dimension, dropout),
            predictor=pdp_predict.NeuralPredictor(device, decimator_dimension, prediction_dimension, edge_dimension,
                                                  meta_data_dimension, mem_hidden_dimension, agg_hidden_dimension,
                                                  mem_agg_hidden_dimension, variable_classifier, function_classifier),
            local_search_iterations=local_search_iterations, epsilon=epsilon)
        self.to(device)


class ReinforceSurveyPropagatorSolver(PropagatorDecimatorSolverBase):
    """The classical Reinforce solver, model type `reinforce` (reference solver.py:598-610): SP with the pi
    reinforcement term, external forces set from the SP biases under a batch-global coin, no variable fixing.  With no
    termination callback or the trainer's, the whole loop runs in one persistent kernel (pdp_set_reinforce); a caller's own
    callback, or a coin source set on the decimator, runs it step by step on the library's stateless operators
    (pdp_sp_step, pdp_score, pdp_edge_aggregate, pdp_cnf_eval)."""

    def __init__(self, device, name, pi=0.1, decimation_probability=0.5, local_search_iterations=0, epsilon=0.05):
        super(ReinforceSurveyPropagatorSolver, self).__init__(
            device=device, name=name,
            propagator=pdp_propagate.SurveyPropagator(device, decimator_dimension=1, include_adaptors=False, pi=pi),
            decimator=pdp_decimate.ReinforceDecimator(
                device, scorer=pdp_predict.SurveyScorer(device, message_dimension=1, include_adaptors=False, pi=pi),
                decimation_probability=decimation_probability),
            predictor=pdp_predict.ReinforcePredictor(device=device),
            local_search_iterations=local_search_iterations, epsilon=epsilon)


class NeuralSequentialDecimatorSolver(PropagatorDecimatorSolverBase):
    """Neural propagator + sequential decimator with a neural scorer, model type `np-d-np` (reference
    solver.py:616-637).  Step by step: dense layers through torch, segmented sums / statistics / variable fixing with
    unit propagation and peeling / CNF check / WalkSAT on the library's kernels."""

    def __init__(self, device, name, edge_dimension, meta_data_dimension, propagator_dimension, decimator_dimension,
                 mem_hidden_dimension, agg_hidden_dimension, mem_agg_hidden_dimension, classifier_dimension, dropout,
                 tolerance, t_max, local_search_iterations=0, epsilon=0.05, decimation_fraction=0.0):
        super(NeuralSequentialDecimatorSolver, self).__init__(
            device=device, name=name,
            propagator=pdp_propagate.NeuralMessagePasser(device, edge_dimension, decimator_dimension, meta_data_dimension,
                                                         propagator_dimension, mem_hidden_dimension, mem_agg_hidden_dimension,
                                                         agg_hidden_dimension, dropout),
            decimator=pdp_decimate.SequentialDecimator(
                device, message_dimension=(3, 1),
                scorer=pdp_predict.NeuralPredictor(device, decimator_dimension, 1, edge_dimension, meta_data_dimension,
                                                   mem_hidden_dimension, agg_hidden_dimension, mem_agg_hidden_dimension,
                                                   variable_classifier=util.PerceptronTanh(decimator_dimension,
                                                                                           classifier_dimension, 1),
                                                   function_classifier=None),
                tolerance=tolerance, t_max=t_max, decimation_fraction=decimation_fraction),
            predictor=pdp_predict.IdentityPredictor(device=device, random_fill=True),
            local_search_iterations=local_search_iterations, epsilon=epsilon)
        self.to(device)
