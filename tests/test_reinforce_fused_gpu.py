"""GPU: model type `reinforce` in the persistent kernel (pdp_set_reinforce) against the C restatement of its loop
(tests/reinforce_oracle.c), the reference's goldens, and the step loop it replaces in ReinforceSurveyPropagatorSolver."""
import json
import os

import numpy as np
import pytest
import torch

from oracle import pdp_oracle as po
from pdp_solver_b200 import cnfgen
from tests import reinforce_oracle as ro
from tests.conftest import GOLDEN, ROOT
from tests.helpers import golden, load, maxdiff, name

pytestmark = pytest.mark.gpu

SURVEY_TOL = 1e-4


def dev():
    return torch.device("cuda:0")


def T(x):
    return torch.from_numpy(np.ascontiguousarray(x)).to(dev())


def C(x):
    return x.detach().cpu().numpy()


def _standard_termination():
    def termination(active, prediction, sat_problem):
        raise RuntimeError("unreachable: evaluated inside the kernel")
    termination._pdp_standard_termination = True
    return termination


def _replicate(batch, b):
    from pdp_solver_b200.nn.solver import SATProblem
    gm, bvm, bfm, ef = (torch.from_numpy(np.ascontiguousarray(x)) for x in batch)
    gm, bvm, bfm, ef, _ = SATProblem._replicate_batch(gm, bvm, bfm, ef.reshape(-1, 1), None, b)
    return gm.numpy(), bvm.numpy(), bfm.numpy(), ef.numpy()


CASES = {
    "3sat": lambda: cnfgen.random_batch(6, 60, 3, 4.0, 501),
    "mixed": lambda: cnfgen.mixed_batch([(40, 3, 4.1), (20, 5, 15.0), (30, 4, 8.5), (50, 3, 3.6)], 502),
}


@pytest.mark.parametrize("case", sorted(CASES))
@pytest.mark.parametrize("check_termination", [True, False], ids=["ct", "noct"])
@pytest.mark.parametrize("rep", [1, 2])
def test_strict_fused_equals_restatement(case, check_termination, rep):
    """strict-math build == the C restatement bit for bit: iterations, freeze iteration per problem, final solution, q
    and [eta, ext]"""
    batch = CASES[case]()
    if rep > 1:
        batch = _replicate(batch, rep)
    gm, bvm, bfm, ef = batch
    E = gm.shape[1]
    iters, pi, p_dec = 60, 0.05, 0.5
    rng = np.random.default_rng(7)
    coins = rng.random(iters, dtype=np.float32)
    init = po.init_state(E, True, rng)
    ro.set_math_mode(True)
    o = ro.ReinforceOracle(gm, bvm, bfm, ef)
    n, merged, freeze, q, f = o.reinforce_run(init[0], init[1], iters, pi, p_dec, coins, check_termination, rep)
    om = o.masks()

    from pdp_solver_b200.engine import Context
    ctx = Context(T(gm), T(bvm), T(bfm), T(ef), strict_math=True)
    ctx.simplify()
    ctx.load_state((T(init[0][0]), T(init[0][1])), (T(init[1][0]), T(init[1][1])))
    ctx.set_reinforce(T(coins), p_dec)
    gn = ctx.sp_run(iters, 0.0, 0, check_termination, rep, pi, full_state=True, sync=True)
    gq, gf = ctx.store_state()
    m = ctx.get_masks()
    _, _, gfreeze = ctx.problem_flags()
    assert gn == n
    assert np.array_equal(C(gfreeze), freeze)
    assert np.array_equal(C(m["sol"]), om["sol"])
    assert np.array_equal(C(gq), q, equal_nan=True)
    assert np.array_equal(C(gf), f, equal_nan=True)
    # every run counts in full against the coins: a further iteration could read past them
    with pytest.raises(Exception):
        ctx.sp_run(1, 0.0, 0, check_termination, rep, pi, full_state=True, sync=True)


def _golden_model(z, W=0):
    from pdp_solver_b200.nn import solver as S
    return S.ReinforceSurveyPropagatorSolver(dev(), "r", pi=float(z["pi"]), decimation_probability=float(z["p_dec"]),
                                             local_search_iterations=W, epsilon=0.5)


def _forward(model, z, check_termination):
    gm, bvm, bfm, ef = T(z["graph_map"]), T(z["bvm"]), T(z["bfm"]), T(z["ef"])
    init = ((T(z["init_p0"]), T(z["init_p1"])), (T(z["init_d0"]), T(z["init_d1"])))
    with torch.no_grad():
        return model(init_state=init, graph_map=gm, batch_variable_map=bvm, batch_function_map=bfm, edge_feature=ef,
                     meta_data=None, is_training=False, iteration_num=int(z["T"]), check_termination=check_termination,
                     simplify=True, batch_replication=1)


@pytest.mark.parametrize("path", golden("reinforce_*.npz"), ids=name)
def test_product_fused_vs_reference(path, monkeypatch):
    """product build, the reference's coins injected through the coin-draw helper (padded with 1.0, a coin that never
    fires): iteration count and final prediction exact, messages within the survey tolerance"""
    from pdp_solver_b200.nn import pdp_decimate
    z = load(path)
    coins = np.concatenate([z["coins"], np.ones(int(z["T"]), np.float32)])[: int(z["T"])].astype(np.float32)
    real = pdp_decimate.draw_coins

    def golden_coins(n, device):
        _, state = real(0, device)
        return T(coins[:n]), state

    monkeypatch.setattr(pdp_decimate, "draw_coins", golden_coins)
    model = _golden_model(z)
    (vp, _), (ps, ds) = _forward(model, z, _standard_termination())
    assert int(model.last_iterations.item()) == z["preds"].shape[0], "iteration count differs"
    assert maxdiff(C(vp).reshape(-1), z["pred"]) == 0
    assert maxdiff(C(ps[0]), z["final_q"]) < SURVEY_TOL and maxdiff(C(ps[1]), z["final_f"]) < SURVEY_TOL
    assert ds[1] is ps[1]


@pytest.mark.parametrize("path", golden("reinforce_*.npz"), ids=name)
@pytest.mark.parametrize("check_termination", [True, False], ids=["ct", "noct"])
def test_fused_equals_step_loop(path, check_termination):
    """same torch.manual_seed, fused vs the step loop (forced by a coin source that draws what _coin draws): the same
    iteration count, the same final prediction after WalkSAT, and the generator left in the same place"""
    z = load(path)
    ct = _standard_termination() if check_termination else None
    out = []
    for fused in (True, False):
        model = _golden_model(z, W=20)
        if not fused:
            model._decimator._coin_source = lambda: torch.rand(1, device=dev()).item()
        torch.manual_seed(99)
        (vp, _), (ps, _) = _forward(model, z, ct)
        out.append((int(model.last_iterations.item()), C(vp).reshape(-1), C(ps[1]), float(torch.rand(1, device=dev()).item())))
    (n0, p0, f0, r0), (n1, p1, f1, r1) = out
    assert n0 == n1
    assert np.array_equal(p0, p1)
    assert r0 == r1
    assert maxdiff(f0, f1) < SURVEY_TOL


def test_cli_reinforce_consistent(tmp_path):
    """satyr.py with config/Predict/reinforce.yaml (fused): every line agrees with the C oracle's CNF check of its solution"""
    from pdp_solver_b200 import satyr
    from pdp_solver_b200.factorgraph.dataset import collate_segment, parse_row
    out = str(tmp_path / "out.json")
    argv = [os.path.join(ROOT, "config", "Predict", "reinforce.yaml"), os.path.join(GOLDEN, "cli_small.json"), "200",
            "-o", out, "-s", "1"]
    assert satyr.main(argv) == 0
    rows = {}
    with open(os.path.join(GOLDEN, "cli_small.json")) as fh:
        for line in fh:
            d = json.loads(line)
            rows[d[4][0]] = d
    lines = [l for l in open(out).read().split("\n") if l]
    assert len(lines) == len(rows)
    for l in lines:
        o = json.loads(l)
        d = rows[o["ID"]]
        gm, bvm, bfm, ef, _, _, _ = collate_segment([parse_row(json.dumps(d))])
        orc = po.Oracle(gm.numpy(), bvm.numpy(), bfm.numpy(), ef.numpy())
        solved, n_unsat = orc.cnf_eval(np.array(o["solution"], dtype=np.float32))
        assert int(np.asarray(solved).reshape(-1)[0]) == o["solved"]
        assert int(np.asarray(n_unsat).reshape(-1)[0]) == o["unsat_clauses"]


def _ctx_run(batch, init, coins, iters, pi, p_dec, ct, rep, strict, generic=False, full_state=False):
    from pdp_solver_b200.engine import Context
    gm, bvm, bfm, ef = batch
    ctx = Context(T(gm), T(bvm), T(bfm), T(ef), strict_math=strict)
    ctx.simplify()
    ctx.load_state((T(init[0][0]), T(init[0][1])), (T(init[1][0]), T(init[1][1])))
    ctx.set_reinforce(T(coins), p_dec)
    n = ctx.sp_run(iters, 0.0, 0, ct, rep, pi, full_state=full_state, generic=generic, sync=True)
    q, f = ctx.store_state()
    m = ctx.get_masks()
    _, _, freeze = ctx.problem_flags()
    return n, C(freeze), C(m["sol"]), C(q), C(f)


def _same(a, b):
    assert a[0] == b[0]
    for x, y in zip(a[1:], b[1:]):
        assert np.array_equal(x, y, equal_nan=True)


BLOCKED_CASES = dict(CASES, big=lambda: cnfgen.random_batch(2, 1000000, 3, 4.2, 503))


@pytest.mark.parametrize("case", sorted(BLOCKED_CASES))
@pytest.mark.parametrize("check_termination", [True, False], ids=["ct", "noct"])
@pytest.mark.parametrize("strict", [True, False], ids=["strictmath", "productmath"])
def test_blocked_equals_generic(case, check_termination, strict):
    """the blocked passes (per-variable pi terms) == the generic passes bit for bit: iterations, freeze iterations, solution,
    and the exported [E,3] / [E,2] state -- both without the full state (q_s, q_* re-derived on export with the forces the
    last sweep read) and against the generic run that tracks the full state"""
    if case == "big" and strict:
        pytest.skip("2 x n = 10^6 in the product build only")
    batch = BLOCKED_CASES[case]()
    E = batch[0].shape[1]
    iters = 12 if case == "big" else 60
    rng = np.random.default_rng(11)
    coins = rng.random(iters, dtype=np.float32)
    init = po.init_state(E, False)
    args = (batch, init, coins, iters, 0.05, 0.5, check_termination, 1, strict)
    blocked = _ctx_run(*args)
    _same(blocked, _ctx_run(*args, generic=True))
    _same(blocked, _ctx_run(*args, generic=True, full_state=True))


def test_mixed_forces_take_the_generic_passes():
    """a loaded state whose forces differ between the edges of a variable: the default run (which must not take the
    blocked passes) equals the generic run bit for bit, and the solver's fused path equals the step loop"""
    batch = CASES["3sat"]()
    E = batch[0].shape[1]
    rng = np.random.default_rng(12)
    init = po.init_state(E, False)
    for st in (init[0][1], init[1][1]):
        st[:, 1] = np.where(rng.random(E) < 0.5, -1.0, 1.0).astype(np.float32)
    coins = rng.random(60, dtype=np.float32)
    args = (batch, init, coins, 60, 0.05, 0.5, True, 1, False)
    _same(_ctx_run(*args), _ctx_run(*args, generic=True))

    from pdp_solver_b200.nn import solver as S
    gm, bvm, bfm, ef = (T(x) for x in batch)
    state = ((T(init[0][0]), T(init[0][1])), (T(init[1][0]), T(init[1][1])))
    out = []
    for fused in (True, False):
        model = S.ReinforceSurveyPropagatorSolver(dev(), "r", pi=0.05, decimation_probability=0.5, local_search_iterations=10)
        if not fused:
            model._decimator._coin_source = lambda: torch.rand(1, device=dev()).item()
        torch.manual_seed(5)
        with torch.no_grad():
            (vp, _), (ps, _) = model(init_state=tuple(tuple(x.clone() for x in s) for s in state), graph_map=gm,
                                     batch_variable_map=bvm, batch_function_map=bfm, edge_feature=ef.reshape(-1, 1),
                                     meta_data=None, is_training=False, iteration_num=60,
                                     check_termination=_standard_termination(), simplify=True)
        out.append((int(model.last_iterations.item()), C(vp).reshape(-1), C(ps[1]), float(torch.rand(1, device=dev()).item())))
    (n0, p0, f0, r0), (n1, p1, f1, r1) = out
    assert n0 == n1 and np.array_equal(p0, p1) and r0 == r1
    assert maxdiff(f0, f1) < SURVEY_TOL
