"""CPU: SP-inspired decimation (a fraction of each problem's active variables fixed per decimation step) in the C oracle
with the fraction rule (tests/sid_oracle.c), against a numpy restatement of the rule (include/pdp_b200.h, pdp_decimation_select), plus the validation of the
fraction in the constructors and the YAML model config."""
import math
import os
import types

import numpy as np
import pytest

from oracle import pdp_oracle as po
from tests.sid_oracle import SidOracle

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def numpy_rule(coeff, score, bvm, B, av, fraction, problem_sel=None):
    """assignment [V]: for every selected problem without NaN coefficients and with a positive coefficient, K = max(1,
    floor(f * active)) variables: K == 1 the first index of the max of fl(fl(c - min) + 1) (util.py:257-265), else the
    first K active variables with c > 0 by (c descending, index ascending)"""
    coeff = np.asarray(coeff, np.float32)
    score = np.asarray(score, np.float32)
    bvm = np.asarray(bvm)
    av = np.asarray(av, np.float32)
    out = np.zeros(coeff.shape[0], np.float32)
    f = float(np.float32(fraction))
    for b in range(B):
        if problem_sel is not None and not problem_sel[b]:
            continue
        idx = np.nonzero(bvm == b)[0]
        c = coeff[idx]
        if np.isnan(c).any() or not (c > 0).any():
            continue
        K = max(1, int(math.floor(f * float(av[idx].sum()))))
        if K == 1:
            key = (c - c.min()).astype(np.float32) + np.float32(1.0)
            j = idx[int(np.argmax(key))]
            out[j] = np.sign(score[j])
        else:
            cand = (c > 0) & (av[idx] > 0)
            ci, cc = idx[cand], c[cand]
            take = ci[np.lexsort((ci, -cc))[:K]]
            out[take] = np.sign(score[take])
    return out


def _batch(sizes, seed=0):
    """a batch of tiny random 3-SAT problems with the given variable counts"""
    from pdp_solver_b200 import cnfgen
    rng = np.random.Generator(np.random.PCG64(seed))
    return cnfgen.collate([(n,) + cnfgen.random_ksat(n, 3, 4.0, rng) for n in sizes])


def crafted():
    """problems: 0 ties (equal c, K above #ties), 1 zeros + inactive variables, 2 a NaN coefficient, 3 K above the
    candidate count, 4 K == 1 (arg-max with the +1 key rounding a tiny difference away), 5 not selected"""
    sizes = [40, 40, 30, 60, 12, 20]
    gm, bvm, bfm, ef = _batch(sizes)
    V = bvm.shape[0]
    ptr = np.concatenate(([0], np.cumsum(sizes)))
    rng = np.random.default_rng(3)
    c = rng.random(V).astype(np.float32)
    score = (rng.random(V).astype(np.float32) - 0.5)
    av = np.ones(V, np.float32)
    p = slice(ptr[0], ptr[1])
    c[p] = np.float32(0.5)
    c[ptr[0] + 7] = np.float32(0.75)
    p1 = np.arange(ptr[1], ptr[2])
    c[p1[::3]] = 0.0
    av[p1[1::4]] = 0.0
    c[p1[1::4]] = 0.0
    c[ptr[2] + 5] = np.nan
    p3 = np.arange(ptr[3], ptr[4])
    c[p3] = 0.0
    c[p3[[4, 9, 33]]] = np.float32(0.25)
    p4 = np.arange(ptr[4], ptr[5])
    c[p4] = np.float32(1e-9)
    c[p4[6]] = np.float32(2e-9)     # fl(fl(c - min) + 1) == 1 for every variable: the first index wins
    score[score == 0] = 0.5
    sel = np.array([1, 1, 1, 1, 1, 0], np.uint8)
    return (gm, bvm, bfm, ef), c, score, av, sel


@pytest.mark.parametrize("fraction", [0.0, 0.02, 0.1, 0.3, 0.9])
def test_select_matches_numpy_rule(fraction):
    batch, c, score, av, sel = crafted()
    o = SidOracle(*batch)
    o.set_masks(av=av)
    B = o.B
    for ps in (sel, None):
        got = o.decimation_select(c, score, fraction, ps)
        want = numpy_rule(c, score, batch[1], B, av, fraction, ps)
        assert np.array_equal(got, want)
    if fraction == 0.1:
        bvm = batch[1]
        got = o.decimation_select(c, score, fraction, sel)
        n = [int((got[bvm == b] != 0).sum()) for b in range(B)]
        assert n[0] == 4 and n[2] == 0 and n[3] == 3 and n[4] == 1 and n[5] == 0
        assert got[np.nonzero(bvm == 4)[0][0]] != 0   # K == 1: key-rounded arg-max, first index


@pytest.mark.parametrize("bad", [-0.1, 1.0, 1.5, float("nan"), float("inf")])
def test_oracle_rejects_bad_fraction(bad):
    batch, c, score, av, sel = crafted()
    o = SidOracle(*batch)
    with pytest.raises(ValueError):
        o.set_decimation_fraction(bad)
    with pytest.raises(ValueError):
        o.decimation_select(c, score, bad)
    strict = SidOracle(*batch, strict=True)
    with pytest.raises(ValueError):
        strict.set_decimation_fraction(0.1)
    strict.set_decimation_fraction(0.0)


@pytest.mark.parametrize("fraction", [0.02, 0.1])
def test_trajectory_fixes_min_k_candidates(fraction):
    """every decimation step of an oracle trajectory takes exactly min(K_b, #candidates) variables of each problem it
    decimates, and they are the numpy rule's choice on that step's scores"""
    from pdp_solver_b200 import cnfgen
    batch = cnfgen.random_batch(6, 300, 3, 4.1, 21)
    gm, bvm = batch[0], batch[1]
    o = SidOracle(*batch)
    o.set_decimation_fraction(fraction)
    o.simplify()
    o.set_state(*po.init_state(gm.shape[1]))
    steps = 0
    for _ in range(150):
        m0 = o.masks()
        n0 = o.trace().shape[0]
        na = o.iterate(0.02, 25, True)
        tr = o.trace()[n0:]
        if tr.shape[0]:
            _, fs = o.state()
            score = o.score(fs, m0["af"])
            coeff = np.abs(score) * m0["av"]
            probs = np.unique(bvm[tr[:, 1]])
            sel = np.zeros(o.B, np.uint8)
            sel[probs] = 1
            want = numpy_rule(coeff, score, bvm, o.B, m0["av"], fraction, sel)
            got = np.zeros(o.V, np.float32)
            got[tr[:, 1]] = tr[:, 2]
            assert np.array_equal(got, want)
            for b in probs:
                idx = bvm == b
                K = max(1, int(math.floor(float(np.float32(fraction)) * float(m0["av"][idx].sum()))))
                ncand = int(((coeff > 0) & (m0["av"] > 0) & idx).sum())
                assert int((bvm[tr[:, 1]] == b).sum()) == min(K, ncand)
            steps += 1
        if na == 0:
            break
    assert steps >= 3, "too few decimation steps: the test does not exercise the rule"


def test_zero_fraction_is_todays_trajectory():
    """f = 0 set explicitly: the reference's golden trajectory, and the same bytes as the oracle's own loop"""
    from tests.helpers import golden, load
    z = load(golden("traj_det_a.npz")[0])
    outs = []
    for sid in (False, True):
        o = (SidOracle if sid else po.Oracle)(z["graph_map"], z["bvm"], z["bfm"], z["ef"], strict=False)
        if sid:
            o.set_decimation_fraction(0.0)
        o.simplify()
        o.set_state((z["init_pq"], z["init_pf"]), (z["init_dq"], z["init_df"]))
        done = o.run(int(z["T"]), float(z["tol"]), float(z["t_max"]), True)
        q, fs = o.state()
        m = o.masks()
        outs.append((np.int64(done), q, fs, m["av"], m["af"], m["sol"], m["active"], o.trace(), o.counters()))
    for a, b in zip(*outs):
        assert np.asarray(a).tobytes() == np.asarray(b).tobytes()
    key = lambda a: a[np.lexsort((a[:, 1], a[:, 0]))]
    assert np.array_equal(key(outs[1][7]), key(z["events"].astype(np.int64)))


@pytest.mark.parametrize("bad", [-0.01, 1.0, float("nan"), float("inf"), "x", None])
def test_constructors_validate(bad):
    from pdp_solver_b200.nn import solver
    with pytest.raises(ValueError):
        solver.SurveyPropagatorSolver("cpu", "m", 0.02, 100, decimation_fraction=bad)


def test_fraction_is_not_in_state_dict():
    from pdp_solver_b200.nn import solver
    ref = solver.SurveyPropagatorSolver("cpu", "m", 0.02, 100)
    sid = solver.SurveyPropagatorSolver("cpu", "m", 0.02, 100, decimation_fraction=0.01)
    assert sid._decimator._decimation_fraction == pytest.approx(0.01) and ref._decimator._decimation_fraction == 0.0
    assert set(ref.state_dict()) == set(sid.state_dict())
    sid.load_state_dict(ref.state_dict(), strict=True)


def _build(config):
    from pdp_solver_b200.trainer import SatFactorGraphTrainer
    fake = types.SimpleNamespace(_device="cpu", _logger=None)
    base = dict(model_name="m", local_search_iteration=0, epsilon=0.05, tolerance=0.02, t_max=100)
    base.update(config)
    return SatFactorGraphTrainer._build_graph(fake, base)[0]


def test_yaml_fraction():
    import yaml
    with open(os.path.join(ROOT, "config", "Predict", "sp.yaml")) as f:
        sp = yaml.safe_load(f)
    with open(os.path.join(ROOT, "config", "Predict", "sp-sid.yaml")) as f:
        sid = yaml.safe_load(f)
    assert set(sid) == set(sp) | {"decimation_fraction"} and all(sid[k] == sp[k] for k in sp)
    model = _build(dict(sid))
    assert model._decimator._decimation_fraction == pytest.approx(sid["decimation_fraction"])
    assert _build(dict(model_type="p-d-p"))._decimator._decimation_fraction == 0.0
    with pytest.raises(ValueError):
        _build(dict(model_type="p-d-p", decimation_fraction=1.0))
    with pytest.raises(ValueError):
        _build(dict(model_type="walk-sat", decimation_fraction=0.05))
    with pytest.raises(ValueError):
        _build(dict(model_type="reinforce", pi=0.1, decimation_probability=0.5, decimation_fraction=0.05))
    _build(dict(model_type="walk-sat", decimation_fraction=0.0))
