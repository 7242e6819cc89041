"""Predict-side drop-in for the reference's `pdp.trainer` (reference src/pdp/trainer.py): builds the solver named by
`model_type` from the YAML model_config, runs it over the input batches and writes one JSON object per problem."""
import numpy as np
import torch
import torch.nn as nn

from .factorgraph import FactorGraphTrainerBase
from .nn import pdp_decimate, solver, util


class Perceptron(nn.Module):
    "The variable classifier of the neural model types (reference trainer.py:20-29); same parameter names."

    def __init__(self, input_dimension, hidden_dimension, output_dimension):
        super(Perceptron, self).__init__()
        self._layer1 = nn.Linear(input_dimension, hidden_dimension)
        self._layer2 = nn.Linear(hidden_dimension, output_dimension, bias=False)

    def forward(self, inp):
        return torch.sigmoid(self._layer2(torch.relu(self._layer1(inp))))


def _bits_to_json_list(bits):
    "uint8 0/1 array -> '[0, 1, 1]' (what str(list_of_ints) gives), without building Python ints"
    n = bits.shape[0]
    if n == 0:
        return "[]"
    buf = np.empty((n, 3), dtype=np.uint8)
    buf[:, 0] = bits + 48
    buf[:, 1] = 44
    buf[:, 2] = 32
    return "[" + buf.tobytes()[:-2].decode("ascii") + "]"


class SatFactorGraphTrainer(FactorGraphTrainerBase):
    "Builds and runs the PDP SAT solvers of the predict path (reference trainer.py:34-162)."

    def __init__(self, config, use_cuda, logger):
        super(SatFactorGraphTrainer, self).__init__(
            config=config, has_meta_data=False, error_dim=config.get("error_dim", 1), loss=None,
            evaluator=nn.L1Loss(), use_cuda=use_cuda, logger=logger)
        self._cnf_evaluator = util.SatCNFEvaluator(device=self._device)
        self._counter = 0

    def _build_graph(self, config):
        "reference trainer.py:48-99"
        t = config["model_type"]
        w, eps = config["local_search_iteration"], config["epsilon"]
        # SP-inspired decimation (optional key): only the model types with a sequential decimator fix variables
        frac = pdp_decimate.check_decimation_fraction(config.get("decimation_fraction", 0.0))
        if frac != 0.0 and t not in ("p-d-p", "np-d-np"):
            raise ValueError("decimation_fraction applies to model types p-d-p and np-d-np only, not %r" % (t,))
        # conflict rollback of SP-inspired decimation (optional key): p-d-p only (np-d-np decimates step-wise on the host)
        rollback = config.get("conflict_rollback", False)
        if rollback is not False and t != "p-d-p":
            raise ValueError("conflict_rollback applies to model type p-d-p only, not %r" % (t,))
        rollback = pdp_decimate.check_conflict_rollback(rollback, frac)
        neural = dict(edge_dimension=config.get("edge_feature_dim"), meta_data_dimension=config.get("meta_feature_dim"),
                      mem_hidden_dimension=config.get("mem_hidden_dim"), agg_hidden_dimension=config.get("agg_hidden_dim"),
                      mem_agg_hidden_dimension=config.get("mem_agg_hidden_dim"), dropout=config.get("dropout", 0),
                      local_search_iterations=w, epsilon=eps)
        if t == "np-nd-np":
            model = solver.NeuralPropagatorDecimatorSolver(
                device=self._device, name=config["model_name"], propagator_dimension=config["hidden_dim"],
                decimator_dimension=config["hidden_dim"], prediction_dimension=config["prediction_dim"],
                variable_classifier=Perceptron(config["hidden_dim"], config["classifier_dim"], config["prediction_dim"]),
                function_classifier=None, **neural)
        elif t == "p-nd-np":
            model = solver.NeuralSurveyPropagatorSolver(
                device=self._device, name=config["model_name"], decimator_dimension=config["hidden_dim"],
                prediction_dimension=config["prediction_dim"],
                variable_classifier=Perceptron(config["hidden_dim"], config["classifier_dim"], config["prediction_dim"]),
                function_classifier=None, **neural)
        elif t == "np-d-np":
            model = solver.NeuralSequentialDecimatorSolver(
                device=self._device, name=config["model_name"], propagator_dimension=config["hidden_dim"],
                decimator_dimension=config["hidden_dim"], classifier_dimension=config["classifier_dim"],
                tolerance=config["tolerance"], t_max=config["t_max"], decimation_fraction=frac, **neural)
        elif t == "p-d-p":
            model = solver.SurveyPropagatorSolver(device=self._device, name=config["model_name"],
                                                  tolerance=config["tolerance"], t_max=config["t_max"],
                                                  local_search_iterations=w, epsilon=eps, decimation_fraction=frac,
                                                  conflict_rollback=rollback)
        elif t == "walk-sat":
            model = solver.WalkSATSolver(device=self._device, name=config["model_name"], iteration_num=w, epsilon=eps)
        elif t == "reinforce":
            model = solver.ReinforceSurveyPropagatorSolver(
                device=self._device, name=config["model_name"], pi=config["pi"],
                decimation_probability=config["decimation_probability"], local_search_iterations=w, epsilon=eps)
        else:
            raise ValueError("unknown model_type %r" % (t,))
        if config.get("verbose"):
            self._logger.info("The model parameter count is %d." % model.parameter_count())
        return [model]

    def _post_process_predictions(self, model, prediction, graph_map, batch_variable_map, batch_function_map,
                                  edge_feature, graph_feat, label, misc_data):
        """One JSON object per problem, the reference's keys, order and text (trainer.py:125-148).  The solution of
        problem i is the slice [ptr[i], ptr[i+1]) of the prediction (the reference selects it with a boolean mask per
        problem: O(B*V))."""
        solved, n_unsat = self._cnf_evaluator(
            variable_prediction=prediction[0], graph_map=graph_map, batch_variable_map=batch_variable_map,
            batch_function_map=batch_function_map, edge_feature=edge_feature, meta_data=graph_feat)
        bits = (prediction[0][:, 0] > 0.5).to(torch.uint8)
        B = solved.shape[0]
        counts = torch.bincount(batch_variable_map.long(), minlength=B)
        bits, solved, n_unsat, counts = bits.cpu().numpy(), solved.cpu().numpy(), n_unsat.cpu().numpy(), counts.cpu().numpy()
        labs = label.detach().cpu().numpy()
        ptr = np.concatenate(([0], np.cumsum(counts)))
        contiguous = bool((np.diff(batch_variable_map.cpu().numpy()) >= 0).all()) if B > 1 else True
        bvm_host = None if contiguous else batch_variable_map.cpu().numpy()
        lines = []
        for i in range(B):
            sol = bits[ptr[i]:ptr[i + 1]] if contiguous else bits[bvm_host == i]
            ident = misc_data[i][0] if len(misc_data[i]) > 0 else ""
            head = str({"ID": ident, "label": int(labs[i, 0]), "solved": int(solved[i].flatten()[0] == 1),
                        "unsat_clauses": int(n_unsat[i].flatten()[0])}).replace("'", '"')
            lines.append(head[:-1] + ', "solution": ' + _bits_to_json_list(sol) + "}\n")
            self._counter += 1
        return "".join(lines)

    def _check_recurrence_termination(self, active, prediction, sat_problem):
        """De-activates the problems already solved (reference trainer.py:150-162).  The solvers recognise this
        method and evaluate it inside the persistent kernel; this body serves any other caller."""
        output, _ = self._cnf_evaluator(
            variable_prediction=prediction[0], graph_map=sat_problem._graph_map,
            batch_variable_map=sat_problem._batch_variable_map, batch_function_map=sat_problem._batch_function_map,
            edge_feature=sat_problem._edge_feature, meta_data=sat_problem._meta_data)
        ok = output[:, 0] > 0.5
        rep = sat_problem._batch_replication
        if rep > 1:
            ok = ok.reshape(rep, -1).any(0).repeat(rep)
        active[(active[:, 0] != 0) & ok, 0] = 0


# the solvers evaluate exactly this method inside the persistent kernel (nn/solver.py _is_standard_termination); an
# override in a subclass is a different function object without the tag and is called iteration by iteration
SatFactorGraphTrainer._check_recurrence_termination._pdp_standard_termination = True
