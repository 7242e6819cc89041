"""CPU: conflict rollback for SP-inspired decimation in the C oracle (tests/rollback_oracle.c): with rollback off it is the
SP-inspired decimation oracle byte for byte; with rollback on, every rollback restores the problem's state from before
the step, h_b equals r_b, and no one-variable step is ever undone.  Plus the validation of the option in the solver
constructor and the YAML model config."""
import math
import os
import types

import numpy as np
import pytest

from oracle import pdp_oracle as po
from tests.rollback_oracle import RollbackOracle
from tests.sid_oracle import SidOracle

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))

# seeded random 3-SAT at alpha = 4.2 whose runs roll back at least once at both fractions: (problems, n, seed)
ROLLBACK_SPECS = [(4, 300, 1), (2, 1000, 3), (6, 200, 5)]


def _run(cls, batch, fraction, T, rollback=None):
    o = cls(*batch)
    o.set_decimation_fraction(fraction)
    if rollback is not None:
        o.set_conflict_rollback(rollback)
    o.simplify()
    o.set_state(*po.init_state(batch[0].shape[1]))
    done = o.run(T, 0.02, 25, True)
    q, fs = o.state()
    m = o.masks()
    return [np.int64(done), q, fs, m["av"], m["af"], m["sol"], m["is_sat"], m["active"], m["em"], o.trace(), o.counters()]


@pytest.mark.parametrize("fraction", [0.0, 0.02, 0.1, 0.3])
def test_rollback_off_is_sid_trajectory(fraction):
    """rollback off: the SP-inspired decimation oracle's trajectory, byte for byte"""
    from pdp_solver_b200 import cnfgen
    batch = cnfgen.random_batch(4, 300, 3, 4.2, 1)
    want = _run(SidOracle, batch, fraction, 150)
    got = _run(RollbackOracle, batch, fraction, 150, rollback=False)
    for a, b in zip(want, got):
        assert np.asarray(a).tobytes() == np.asarray(b).tobytes()


@pytest.mark.parametrize("fraction", [0.1, 0.3])
@pytest.mark.parametrize("spec", ROLLBACK_SPECS, ids=lambda s: "B%d_n%d_s%d" % s)
def test_rollback_restores_state(spec, fraction):
    """step by step: a problem whose rollback count grows in an iteration ends it with the av / af / sol / is_sat it
    started with (masks change only in the decimation step), that step took K_b >= 2 variables, and h_b == r_b"""
    from pdp_solver_b200 import cnfgen
    Bn, n, seed = spec
    batch = cnfgen.random_batch(Bn, n, 3, 4.2, seed)
    bvm, bfm = batch[1], batch[2]
    o = RollbackOracle(*batch)
    o.set_decimation_fraction(fraction)
    o.set_conflict_rollback(True)
    o.simplify()
    o.set_state(*po.init_state(batch[0].shape[1]))
    f = float(np.float32(fraction))
    seen = 0
    for it in range(1, 301):
        h0, r0, _ = o.rollbacks()
        m0 = o.masks()
        n0 = o.trace().shape[0]
        na = o.iterate(0.02, 25, True)
        h1, r1, last1 = o.rollbacks()
        m1 = o.masks()
        assert np.array_equal(h1, r1)
        tr = o.trace()[n0:]
        for b in np.nonzero(r1 > r0)[0]:
            assert r1[b] == r0[b] + 1 and last1[b] == it
            vb, fb = bvm == b, bfm == b
            for k, sel in (("av", vb), ("af", fb), ("sol", vb)):
                assert np.array_equal(m1[k][sel], m0[k][sel]), k
            assert m1["is_sat"][b] == m0["is_sat"][b] and m0["is_sat"][b] != 0
            K = max(1, int(math.floor(f * float(m0["av"][vb].sum()))) >> int(h0[b]))
            assert K >= 2, "a one-variable step was rolled back"
            assert int((bvm[tr[:, 1]] == b).sum()) >= 2   # the trace keeps the undone fixes
            seen += 1
        if na == 0:
            break
    assert seen > 0, "no rollback: the test does not exercise the path"


@pytest.mark.parametrize("bad", [1, "yes", None, 0.5])
def test_constructor_validates(bad):
    from pdp_solver_b200.nn import solver
    with pytest.raises(ValueError):
        solver.SurveyPropagatorSolver("cpu", "m", 0.02, 100, decimation_fraction=0.01, conflict_rollback=bad)
    with pytest.raises(ValueError):   # rollback needs a fraction
        solver.SurveyPropagatorSolver("cpu", "m", 0.02, 100, conflict_rollback=True)


def test_rollback_is_not_in_state_dict():
    from pdp_solver_b200.nn import solver
    ref = solver.SurveyPropagatorSolver("cpu", "m", 0.02, 100)
    rb = solver.SurveyPropagatorSolver("cpu", "m", 0.02, 100, decimation_fraction=0.01, conflict_rollback=True)
    assert rb._decimator._conflict_rollback is True and ref._decimator._conflict_rollback is False
    assert set(ref.state_dict()) == set(rb.state_dict())
    rb.load_state_dict(ref.state_dict(), strict=True)


def _build(config):
    from pdp_solver_b200.trainer import SatFactorGraphTrainer
    fake = types.SimpleNamespace(_device="cpu", _logger=None)
    base = dict(model_name="m", local_search_iteration=0, epsilon=0.05, tolerance=0.02, t_max=100)
    base.update(config)
    return SatFactorGraphTrainer._build_graph(fake, base)[0]


def test_yaml_rollback():
    import yaml
    with open(os.path.join(ROOT, "config", "Predict", "sp-sid.yaml")) as f:
        sid = yaml.safe_load(f)
    with open(os.path.join(ROOT, "config", "Predict", "sp-sid-rollback.yaml")) as f:
        rb = yaml.safe_load(f)
    assert set(rb) == set(sid) | {"conflict_rollback"} and all(rb[k] == sid[k] for k in sid) and rb["conflict_rollback"] is True
    assert _build(dict(rb))._decimator._conflict_rollback is True
    assert _build(dict(sid))._decimator._conflict_rollback is False
    with pytest.raises(ValueError):
        _build(dict(model_type="p-d-p", conflict_rollback=True))   # no fraction
    with pytest.raises(ValueError):
        _build(dict(model_type="p-d-p", decimation_fraction=0.01, conflict_rollback="true"))
    with pytest.raises(ValueError):
        _build(dict(model_type="walk-sat", conflict_rollback=True))
    npdnp = dict(model_type="np-d-np", hidden_dim=4, classifier_dim=4, edge_feature_dim=1, meta_feature_dim=0,
                 mem_hidden_dim=4, agg_hidden_dim=4, mem_agg_hidden_dim=4, decimation_fraction=0.01)
    with pytest.raises(ValueError):
        _build(dict(npdnp, conflict_rollback=True))
