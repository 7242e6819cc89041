"""GPU: SP-inspired decimation (pdp_set_decimation_fraction / pdp_decimation_select) against the C oracle and the numpy
restatement of the rule, and the decimation paths of the fused loop against each other."""
import math

import numpy as np
import pytest
import torch

from tests.test_sid_oracle import crafted, numpy_rule

pytestmark = pytest.mark.gpu


def T(x):
    return torch.from_numpy(np.ascontiguousarray(x)).to("cuda:0")


def C(t):
    return t.detach().cpu().numpy()


def _sorted(tr):
    tr = np.asarray(tr, np.int64)
    return tr[np.lexsort((tr[:, 2], tr[:, 1], tr[:, 0]))]


@pytest.mark.parametrize("fraction", [0.0, 0.02, 0.1, 0.3])
def test_decimation_select_matches_numpy_rule(fraction):
    """crafted vectors (ties, zeros, inactive variables, NaN, K above the candidate count, K == 1) and a batch with one
    40 000-variable problem with forced ties"""
    from pdp_solver_b200 import cnfgen
    from pdp_solver_b200.engine import Context
    batch, c, score, av, sel = crafted()
    ctx = Context(T(batch[0]), T(batch[1]), T(batch[2]), T(batch[3]))
    ctx.set_masks(av=T(av))
    for ps in (sel, None):
        got = C(ctx.decimation_select(T(c), T(score), fraction, None if ps is None else T(ps)))
        assert np.array_equal(got, numpy_rule(c, score, batch[1], ctx.B, av, fraction, ps))
    big = cnfgen.mixed_batch([(40000, 3, 4.2), (300, 3, 4.0), (5000, 3, 4.1)], 5)
    ctx = Context(T(big[0]), T(big[1]), T(big[2]), T(big[3]))
    rng = np.random.default_rng(9)
    V = big[1].shape[0]
    c = np.round(rng.random(V) * 64).astype(np.float32) / 64     # many exact ties
    score = rng.standard_normal(V).astype(np.float32)
    got = C(ctx.decimation_select(T(c), T(score), fraction))
    assert np.array_equal(got, numpy_rule(c, score, big[1], ctx.B, np.ones(V, np.float32), fraction))


def _gpu_run(batch, init, Tn, fraction, strict_math=False, **kw):
    from pdp_solver_b200.engine import Context
    ctx = Context(T(batch[0]), T(batch[1]), T(batch[2]), T(batch[3]), strict_math=strict_math)
    ctx.set_decimation_fraction(fraction)
    ctx.enable_trace(1 << 20)
    ctx.simplify()
    ctx.load_state((T(init[0][0]), T(init[0][1])), (T(init[1][0]), T(init[1][1])))
    done = ctx.sp_run(Tn, 0.02, 25, True, sync=True, **kw)
    q, fs = ctx.store_state()
    m = ctx.get_masks()
    flags, counters, freeze = ctx.problem_flags()
    return dict(done=np.int64(done), tr=_sorted(C(ctx.trace())), av=C(m["av"]), af=C(m["af"]), sol=C(m["sol"]),
                active=C(m["active"]), is_sat=C(m["is_sat"]), flags=C(flags), counters=C(counters), freeze=C(freeze),
                q=C(q[:, 0]), fs=C(fs[:, 0]))


SPECS = [(96, 100, 3, 4.2, 200, 41), (12, 400, 3, 4.0, 150, 42), (40, 60, 3, 3.5, 150, 43)]


def _spec_batch(spec):
    from pdp_solver_b200 import cnfgen
    if spec == "mixed":
        return cnfgen.mixed_batch([(40000, 3, 4.2), (300, 3, 4.0), (1000, 3, 4.1), (150, 3, 3.9)], 61), 150
    Bn, n, k, alpha, Tn, seed = spec
    return cnfgen.random_batch(Bn, n, k, alpha, seed), Tn


@pytest.mark.parametrize("fraction", [0.02, 0.1, 0.3])
@pytest.mark.parametrize("spec", SPECS + ["mixed"], ids=lambda s: s if isinstance(s, str) else "B%d_n%d" % (s[0], s[1]))
def test_strict_build_equals_oracle(spec, fraction):
    """the strict-math build against the oracle, bit for bit: sorted decimation events, masks, solution, flags-level
    verdicts, counters of active problems, iteration count"""
    from oracle import pdp_oracle as po
    from tests import sid_oracle
    batch, Tn = _spec_batch(spec)
    init = po.init_state(batch[0].shape[1])
    sid_oracle.set_math_mode(True)
    try:
        o = sid_oracle.SidOracle(*batch)
        o.set_decimation_fraction(fraction)
        o.simplify()
        o.set_state(*init)
        done = o.run(Tn, 0.02, 25, True)
        om, ref, oc = o.masks(), _sorted(o.trace()), o.counters()
    finally:
        sid_oracle.set_math_mode(False)
    g = _gpu_run(batch, init, Tn, fraction, strict_math=True)
    assert g["done"] == done
    assert ref.shape[0] > 0 and g["tr"].shape == ref.shape and np.array_equal(g["tr"], ref)
    for k in ("av", "af", "active"):
        assert np.array_equal(g[k], om[k]), k
    assert np.array_equal(g["sol"], om["sol"]) and np.array_equal(g["is_sat"], om["is_sat"])
    act = om["active"].astype(bool)
    assert np.array_equal(g["counters"][act], oc[act].astype(np.int32))


@pytest.mark.parametrize("spec", SPECS + ["mixed"], ids=lambda s: s if isinstance(s, str) else "B%d_n%d" % (s[0], s[1]))
def test_all_paths_identical(spec, monkeypatch):
    """f = 0.1: CTA-local, grid-wide with the frontier closure, grid-wide with the full-scan closure, frontier lists of 8
    entries (overflow -> full scans), generic passes: identical results, bit for bit"""
    from oracle import pdp_oracle as po
    batch, Tn = _spec_batch(spec)
    init = po.init_state(batch[0].shape[1])
    outs = []
    for kw, cap in ((dict(), None), (dict(grid_decimation=True), None), (dict(grid_decimation=True, full_closure=True), None),
                    (dict(grid_decimation=True), "8"), (dict(generic=True), None)):
        if cap is None:
            monkeypatch.delenv("PDP_B200_FR_CAP", raising=False)
        else:
            monkeypatch.setenv("PDP_B200_FR_CAP", cap)
        outs.append(_gpu_run(batch, init, Tn, 0.1, **kw))
    assert outs[0]["tr"].shape[0] > 0
    for other in outs[1:]:
        for k in outs[0]:
            assert np.array_equal(outs[0][k], other[k], equal_nan=True), k


def test_full_size_paths():
    """2 x n = 1 000 000 at f = 0.01: the product path equals the full-scan closure and the generic passes bit for bit;
    at least 10 decimation steps, each taking K_b = floor(0.01 * active) variables of the problem (candidates abound)"""
    from pdp_solver_b200 import cnfgen
    from pdp_solver_b200.engine import Context
    batch = cnfgen.random_batch(2, 1000000, 3, 4.2, 123)
    outs = []
    for kw in (dict(), dict(full_closure=True), dict(generic=True, full_closure=True)):
        ctx = Context(T(batch[0]), T(batch[1]), T(batch[2]), T(batch[3]), batch_size=2)
        ctx.set_decimation_fraction(0.01)
        ctx.enable_trace(1 << 21)
        ctx.simplify()
        n0 = C(ctx.get_masks()["av"]).reshape(2, -1).sum(1)
        ctx.load_state_const(1.0 / 3.0, 1.0 / 3.0, 1.0 / 3.0, 0.5, 0.0)
        done = ctx.sp_run(170, 0.02, 100, True, sync=True, **kw)
        m = ctx.get_masks()
        _, counters, _ = ctx.problem_flags()
        outs.append(dict(done=np.int64(done), tr=_sorted(C(ctx.trace())), av=C(m["av"]), af=C(m["af"]), sol=C(m["sol"]),
                         active=C(m["active"]), counters=C(counters)))
        del ctx
    tr = outs[0]["tr"]
    prob = tr[:, 1] // 1000000
    steps = np.unique(tr[:, 0])
    assert steps.shape[0] >= 10, "too few decimation steps: the test does not exercise the regime"
    first = tr[tr[:, 0] == steps[0]]
    for b in (0, 1):   # first step of each problem: K = floor(0.01 * active variables after simplify)
        nb = int((first[:, 1] // 1000000 == b).sum())
        assert nb in (0, int(math.floor(float(np.float32(0.01)) * float(n0[b]))))
    assert prob.max() <= 1
    for other in outs[1:]:
        for k in outs[0]:
            assert np.array_equal(outs[0][k], other[k], equal_nan=True), k


def test_solver_zero_fraction_same_bytes():
    """SurveyPropagatorSolver(decimation_fraction=0.0) gives the bytes of the default solver"""
    from pdp_solver_b200 import cnfgen
    from pdp_solver_b200.nn import solver
    batch = cnfgen.random_batch(16, 300, 3, 4.1, 17)
    outs = []
    for kw in (dict(), dict(decimation_fraction=0.0)):
        torch.manual_seed(0)
        s = solver.SurveyPropagatorSolver("cuda:0", "m", 0.02, 25, local_search_iterations=50, **kw)
        gm, bvm, bfm, ef = (T(x) for x in batch)
        init = s.get_init_state(gm, bvm, bfm, ef.reshape(-1, 1), None, False)
        pred, _ = s(init, gm, bvm, bfm, ef.reshape(-1, 1), None, is_training=False, iteration_num=150)
        outs.append((C(pred[0]), C(s.last_problem._ctx.get_masks()["av"])))
    for a, b in zip(*outs):
        assert a.tobytes() == b.tobytes()


def test_cli_sid_config(tmp_path):
    """satyr.py config/Predict/sp-sid.yaml: every line's verdict agrees with the C oracle's CNF check of its solution"""
    from tests.test_cli_gpu import _check_consistent, _problems, _run_cli
    lines = _run_cli(tmp_path, ["-w", "100"], config="sp-sid.yaml")
    rows = _problems()
    assert len(lines) == len(rows)
    _check_consistent(lines, rows)


def _npdnp(z, fraction):
    from pdp_solver_b200.nn import solver as S
    H, MH, AH, MAH, CH = [int(x) for x in z["dims"]]
    model = S.NeuralSequentialDecimatorSolver("cuda:0", "m", edge_dimension=1, meta_data_dimension=0, propagator_dimension=H,
                                              decimator_dimension=H, mem_hidden_dimension=MH, agg_hidden_dimension=AH,
                                              mem_agg_hidden_dimension=MAH, classifier_dimension=CH, dropout=0,
                                              tolerance=float(z["tol"]), t_max=int(z["t_max"]), local_search_iterations=0,
                                              epsilon=0.5, decimation_fraction=fraction)
    sd = {k[2:]: torch.from_numpy(z[k]) for k in z.files if k.startswith("w:")}
    for pair in str(z["w_alias"]).split(";"):
        if pair:
            k, src = pair.split("=")
            sd[k] = sd[src]
    model.load_state_dict(sd, strict=True)
    model = model.to("cuda:0").eval()
    gm, bvm, bfm, ef = T(z["graph_map"]), T(z["bvm"]), T(z["bfm"]), T(z["ef"])
    model.get_init_state(gm, bvm, bfm, ef, None, randomized=False, batch_replication=1)
    init = ((T(z["init_p0"]), T(z["init_p1"])), (T(z["init_d0"]), T(z["init_d1"])))
    with torch.no_grad():
        model(init_state=init, graph_map=gm, batch_variable_map=bvm, batch_function_map=bfm, edge_feature=ef, meta_data=None,
              is_training=False, iteration_num=int(z["T"]), check_termination=None, simplify=True, batch_replication=1)
    return [(C(i).tolist(), C(s).tolist()) for i, s in model._decimator.decimation_log]


def test_npdnp_fraction(monkeypatch):
    """np-d-np: with every K_b = 1 the decimation log is the f = 0 one; with f = 0.1 every step is the numpy rule on that
    step's coefficients (captured at the stateless selection)"""
    from pdp_solver_b200.engine import Context
    from tests.helpers import golden, load
    z = load(golden("npdnp_a.npz")[0])
    base = _npdnp(z, 0.0)
    assert len(base) > 0
    assert _npdnp(z, 1e-7) == base
    seen = []
    orig = Context.decimation_select

    def spy(self, coeff, score, fraction, problem_sel=None):
        out = orig(self, coeff, score, fraction, problem_sel)
        seen.append((C(coeff), C(score), None if problem_sel is None else C(problem_sel), C(self.get_masks()["av"]), C(out),
                     C(self._bvm), self.B))
        return out

    monkeypatch.setattr(Context, "decimation_select", spy)
    log = _npdnp(z, 0.1)
    assert len(seen) > 0 and len(log) > 0
    for coeff, score, sel, av, out, bvm, B in seen:
        # av after the call: the step's selection has not been applied yet (set_variables follows)
        assert np.array_equal(out, numpy_rule(coeff, score, bvm, B, av, 0.1, sel))
    taken = [sorted(np.nonzero(s[4])[0].tolist()) for s in seen if np.any(s[4])]
    assert [sorted(i) for i, _ in log] == taken
