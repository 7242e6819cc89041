"""GPU: conflict rollback for SP-inspired decimation (pdp_set_conflict_rollback) against the C oracle
(tests/rollback_oracle.c), the decimation paths of the fused loop against each other with rollback on, and the solver and
CLI front ends."""
import numpy as np
import pytest
import torch

from tests.test_sid_gpu import SPECS, C, T, _sorted, _spec_batch

pytestmark = pytest.mark.gpu

FLAG_UP_CONFLICT, FLAG_ROLLED_BACK = 8, 16


def _gpu_run(batch, init, Tn, fraction, strict_math=False, rollback=True, batch_size=None, **kw):
    from pdp_solver_b200.engine import Context
    ctx = Context(T(batch[0]), T(batch[1]), T(batch[2]), T(batch[3]), batch_size=batch_size, strict_math=strict_math)
    ctx.set_decimation_fraction(fraction)
    if rollback:
        ctx.enable_conflict_rollback()
    ctx.enable_trace(1 << 21)
    ctx.simplify()
    if init is None:
        ctx.load_state_const(1.0 / 3.0, 1.0 / 3.0, 1.0 / 3.0, 0.5, 0.0)
    else:
        ctx.load_state((T(init[0][0]), T(init[0][1])), (T(init[1][0]), T(init[1][1])))
    done = ctx.sp_run(Tn, 0.02, 25, True, sync=True, **kw)
    q, fs = ctx.store_state()
    m = ctx.get_masks()
    flags, counters, freeze = ctx.problem_flags()
    count, last = ctx.rollbacks()
    out = dict(done=np.int64(done), tr=_sorted(C(ctx.trace())), av=C(m["av"]), af=C(m["af"]), sol=C(m["sol"]),
               active=C(m["active"]), is_sat=C(m["is_sat"]), flags=C(flags), counters=C(counters), freeze=C(freeze),
               q=C(q[:, 0]), fs=C(fs[:, 0]), count=C(count), last=C(last))
    return out, ctx


def _check_consistent(g, ctx):
    """flag bits agree with the counts, the layout self-check is clean and the edge-mask bits follow the node masks"""
    assert np.array_equal((g["flags"] & FLAG_ROLLED_BACK) != 0, g["count"] > 0)
    assert np.array_equal((g["flags"] & FLAG_UP_CONFLICT) != 0, g["is_sat"] == 0)
    errs, info = ctx.check_layout()
    if info["blocked"]:
        E = ctx.E
        assert errs[:6] == [0] * 6 and errs[6] == E and errs[7] == E, errs
    else:
        assert errs[:6] == [0] * 6, errs
    assert ctx.check_edge_mask() == [0, 0]


@pytest.mark.parametrize("fraction", [0.1, 0.3])
@pytest.mark.parametrize("spec", SPECS + ["mixed"], ids=lambda s: s if isinstance(s, str) else "B%d_n%d" % (s[0], s[1]))
def test_strict_build_equals_oracle(spec, fraction):
    """the strict-math build against the rollback oracle, bit for bit: sorted decimation events (undone fixes included),
    masks, solution, is_sat, rollback counts and iterations, iteration count"""
    from oracle import pdp_oracle as po
    from tests import rollback_oracle
    batch, Tn = _spec_batch(spec)
    init = po.init_state(batch[0].shape[1])
    rollback_oracle.set_math_mode(True)
    try:
        o = rollback_oracle.RollbackOracle(*batch)
        o.set_decimation_fraction(fraction)
        o.set_conflict_rollback(True)
        o.simplify()
        o.set_state(*init)
        done = o.run(Tn, 0.02, 25, True)
        om, ref, oc = o.masks(), _sorted(o.trace()), o.counters()
        oh, orr, olast = o.rollbacks()
    finally:
        rollback_oracle.set_math_mode(False)
    g, ctx = _gpu_run(batch, init, Tn, fraction, strict_math=True)
    assert g["done"] == done
    assert ref.shape[0] > 0 and g["tr"].shape == ref.shape and np.array_equal(g["tr"], ref)
    for k in ("av", "af", "active"):
        assert np.array_equal(g[k], om[k]), k
    assert np.array_equal(g["sol"], om["sol"]) and np.array_equal(g["is_sat"], om["is_sat"])
    act = om["active"].astype(bool)
    assert np.array_equal(g["counters"][act], oc[act].astype(np.int32))
    assert np.array_equal(g["count"], orr.astype(np.int32)) and np.array_equal(g["last"], olast.astype(np.int32))
    if not (spec == "mixed" and fraction == 0.1):   # (the one pairing whose oracle run has no rollback)
        assert orr.sum() > 0, "no rollback: the test does not exercise the path"
    _check_consistent(g, ctx)


_PATHS = ((dict(), None), (dict(grid_decimation=True), None), (dict(grid_decimation=True, full_closure=True), None),
          (dict(grid_decimation=True), "8"), (dict(generic=True), None))


@pytest.mark.parametrize("spec", SPECS + ["mixed"], ids=lambda s: s if isinstance(s, str) else "B%d_n%d" % (s[0], s[1]))
def test_all_paths_identical(spec, monkeypatch):
    """f = 0.3 with rollback: CTA-local, grid-wide with the frontier closure, grid-wide with the full-scan closure, frontier
    lists of 8 entries (overflow -> full scans), generic passes: identical results, bit for bit"""
    from oracle import pdp_oracle as po
    batch, Tn = _spec_batch(spec)
    init = po.init_state(batch[0].shape[1])
    outs = []
    for kw, cap in _PATHS:
        if cap is None:
            monkeypatch.delenv("PDP_B200_FR_CAP", raising=False)
        else:
            monkeypatch.setenv("PDP_B200_FR_CAP", cap)
        g, ctx = _gpu_run(batch, init, Tn, 0.3, **kw)
        _check_consistent(g, ctx)
        outs.append(g)
        del ctx
    assert outs[0]["tr"].shape[0] > 0 and outs[0]["count"].sum() > 0
    for other in outs[1:]:
        for k in outs[0]:
            assert np.array_equal(outs[0][k], other[k], equal_nan=True), k


def test_batch_replication_paths():
    """batch_replication = 2 (grid-wide decimation only): frontier, full-scan and generic passes agree, with rollbacks"""
    from oracle import pdp_oracle as po
    from pdp_solver_b200 import cnfgen
    one = cnfgen.random_batch(12, 300, 3, 4.2, 44)
    gm, bvm, bfm, ef = one
    V, F, B = bvm.shape[0], bfm.shape[0], 12
    batch = (np.concatenate([gm, gm + np.array([[V], [F]], gm.dtype)], 1), np.concatenate([bvm, bvm + B]),
             np.concatenate([bfm, bfm + B]), np.concatenate([ef, ef]))
    init = po.init_state(batch[0].shape[1])
    outs = []
    for kw in (dict(), dict(full_closure=True), dict(generic=True)):
        g, ctx = _gpu_run(batch, init, 200, 0.3, batch_replication=2, **kw)
        _check_consistent(g, ctx)
        outs.append(g)
        del ctx
    assert outs[0]["count"].sum() > 0
    for other in outs[1:]:
        for k in outs[0]:
            assert np.array_equal(outs[0][k], other[k], equal_nan=True), k


def test_full_size_paths():
    """2 x n = 1 000 000 at f = 0.04 with rollback: the product path equals the full-scan closure and the generic passes
    bit for bit, with at least one rollback (they come late: decimation at this size ends after about 1 400 iterations)"""
    from pdp_solver_b200 import cnfgen
    batch = cnfgen.random_batch(2, 1000000, 3, 4.2, 123)
    outs = []
    for kw in (dict(), dict(full_closure=True), dict(generic=True, full_closure=True)):
        g, ctx = _gpu_run(batch, None, 2000, 0.04, batch_size=2, **kw)
        _check_consistent(g, ctx)
        for k in ("q", "fs", "freeze"):
            g.pop(k)
        outs.append(g)
        del ctx
        torch.cuda.empty_cache()
    assert outs[0]["count"].sum() > 0, "no rollback: the test does not exercise the path"
    for other in outs[1:]:
        for k in outs[0]:
            assert np.array_equal(outs[0][k], other[k], equal_nan=True), k


def test_solver_rollback_off_same_bytes():
    """SurveyPropagatorSolver(conflict_rollback=False) gives the bytes of the solver without the keyword"""
    from pdp_solver_b200 import cnfgen
    from pdp_solver_b200.nn import solver
    batch = cnfgen.random_batch(16, 300, 3, 4.1, 17)
    outs = []
    for kw in (dict(decimation_fraction=0.1), dict(decimation_fraction=0.1, conflict_rollback=False)):
        torch.manual_seed(0)
        s = solver.SurveyPropagatorSolver("cuda:0", "m", 0.02, 25, local_search_iterations=50, **kw)
        gm, bvm, bfm, ef = (T(x) for x in batch)
        init = s.get_init_state(gm, bvm, bfm, ef.reshape(-1, 1), None, False)
        pred, _ = s(init, gm, bvm, bfm, ef.reshape(-1, 1), None, is_training=False, iteration_num=150)
        outs.append((C(pred[0]), C(s.last_problem._ctx.get_masks()["av"])))
    for a, b in zip(*outs):
        assert a.tobytes() == b.tobytes()


def test_cli_rollback_config(tmp_path):
    """satyr.py config/Predict/sp-sid-rollback.yaml: every line's verdict agrees with the C oracle's CNF check of its
    solution"""
    from tests.test_cli_gpu import _check_consistent as cli_consistent, _problems, _run_cli
    lines = _run_cli(tmp_path, ["-w", "100"], config="sp-sid-rollback.yaml")
    rows = _problems()
    assert len(lines) == len(rows)
    cli_consistent(lines, rows)
