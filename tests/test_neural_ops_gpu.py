"""The device operators of the neural model types (p-nd-np, np-nd-np, np-d-np) against the float64 restatements of
tests/neural_reference.py, at the shapes where their kernels branch:

- pdp_edge_mlp_forward / pdp_edge_gru_forward (tcgen05 dense layer and GRU cell): output widths around the 16-column
  groups and the 256-column pass, K around the 16-element chunks, one to three row sources with boundaries inside a
  half chunk and 4-byte storage offsets, one and several 128-row tiles per CTA, one to three GRU passes; bitwise
  invariances under row order, ring depth and store path;
- pdp_edge_aggregate: bit for bit the sequential fp32 sum in ascending edge order, as the header states;
- pdp_sp_step_adapted: bit for bit pdp_sp_step in the strict-math build, within an fp64 bound in the product build;
- the whole neural models at the reference's dimensions, tcgen05 against the library GEMMs."""
import ctypes

import numpy as np
import pytest
import torch

from tests import neural_reference as NR

pytestmark = pytest.mark.gpu

# largest observed |error| / tolerance per operator, printed at the end of the module (pytest -s)
WORST = {}


@pytest.fixture(scope="module", autouse=True)
def _report_worst():
    yield
    for k in sorted(WORST):
        print("max error / tolerance  %-14s %.3f" % (k, WORST[k]))


def _note(op, err, tol):
    err, tol = np.broadcast_arrays(np.abs(err), tol)
    live = tol > 0                                  # (frozen rows: tolerance 0, checked for equality separately)
    r = float((err[live] / tol[live]).max()) if live.any() else 0.0
    WORST[op] = max(WORST.get(op, 0.0), r)
    return r


def dev():
    return torch.device("cuda:0")


def sms():
    return torch.cuda.get_device_properties(0).multi_processor_count


def rows_of(spec):
    "row counts by name: one tile per CTA, one more row, >= 3 tiles per CTA with a partial last tile"
    if isinstance(spec, int):
        return spec
    return {"sms128": sms() * 128, "sms128+1": sms() * 128 + 1, "3sms128+17": 3 * sms() * 128 + 17}[spec]


def on_device(a, offset=False):
    """a float32 copy of `a` on the device; offset=True: a view that starts one float into its storage (4-byte aligned
    only), the form a slice like storage[1:] hands a kernel"""
    a = np.ascontiguousarray(a, np.float32)
    if not offset:
        return torch.from_numpy(a).to(dev())
    buf = torch.empty(a.size + 1, dtype=torch.float32, device=dev())
    v = buf[1:].view(a.shape)
    v.copy_(torch.from_numpy(a))
    assert v.is_contiguous() and v.data_ptr() % 8 == 4
    return v


def C(t):
    return t.detach().cpu().numpy()


# ---------------------------------------------------------------------------------------------------------------------
# dense layer
# ---------------------------------------------------------------------------------------------------------------------
def _linear_case(rows, pieces, n_out, act=1, mask="binary", offsets=(), bias=True, seed=0):
    from pdp_solver_b200.nn import tensor_ops as TO
    K = sum(pieces)
    torch.manual_seed(seed)
    lin = torch.nn.Linear(K, n_out, bias=bias).to(dev())
    w = C(lin.weight)
    b = C(lin.bias) if bias else None
    rng = np.random.default_rng(seed)
    x = NR.coherent_rows(rng.standard_normal((rows, K)).astype(np.float32), w, -8.0) if rows else np.zeros((0, K), np.float32)
    cuts = np.cumsum([0] + list(pieces))
    src = [on_device(x[:, cuts[i]:cuts[i + 1]], i in offsets) for i in range(len(pieces))]
    m = {"none": None, "binary": (rng.random(rows) > 0.2).astype(np.float32), "fraction": rng.random(rows).astype(np.float32)}[mask]
    out = TO.TensorLinear(lin)(src, act=act, row_mask=None if m is None else on_device(m))
    assert out.shape == (rows, n_out)
    ref, tol = NR.linear64(x, w, b, act, m)
    got = C(out).astype(np.float64)
    assert (np.abs(got - ref) <= tol).all(), "max error/tol %.2f" % _note("linear", got - ref, tol)
    _note("linear", got - ref, tol)
    if m is not None and mask == "binary":
        assert (C(out)[m == 0] == 0).all()
    return lin, src, out


# (rows, pieces, n_out, act, mask, offsets): the branch each case reaches is in its id
LINEAR_CASES = (
    # output width: odd n_out -> scalar stores; n_out * 4 % 16 != 0 -> tail of the tile's bulk store (1001 rows: the last
    # tile has 105); 256 -> one full 256-column MMA
    [("n%d" % n, (1001, (150, 1), n, n % 2, "binary", ())) for n in NR.LINEAR_N_OUT] +
    # K: below one chunk, around 16, odd, 19 chunks, the 64-chunk limit (single source; odd K -> element path)
    [("K%d" % k, (1001, (k,), 100, 1, "fraction", ())) for k in NR.LINEAR_K] +
    [
        ("three_pieces_100_50_1", (1001, (100, 50, 1), 100, 1, "binary", ())),
        ("three_pieces_inside_half_chunks_5_13_3", (1001, (5, 13, 3), 50, 0, "none", ())),
        ("odd_widths_75_75_1", (1001, (75, 75, 1), 100, 1, "binary", ())),
        ("row_150_copy_16_8_8", (1001, (150,), 150, 0, "none", ())),
        ("offset_piece0_s_cd_element_path", (1001, (150, 1), 100, 1, "binary", (0,))),
        ("offset_piece1_of_three", (1001, (100, 50, 1), 100, 0, "fraction", (1,))),
        ("offset_all_pieces", (1001, (64, 36, 51), 17, 1, "none", (0, 1, 2))),
    ] +
    [("rows%s" % r, (r, (150, 1), 100, 1, "fraction", ())) for r in (0, 1, 127, 128, 129, "sms128", "sms128+1", "3sms128+17")]
)


@pytest.mark.parametrize("case", [c for _, c in LINEAR_CASES], ids=[i for i, _ in LINEAR_CASES])
def test_linear_vs_fp64(case):
    rows, pieces, n_out, act, mask, offsets = case
    _linear_case(rows_of(rows), pieces, n_out, act, mask, offsets, bias=(n_out != 50), seed=n_out + sum(pieces))


def test_linear_rejects_what_does_not_fit():
    from pdp_solver_b200 import _lib
    from pdp_solver_b200.nn import tensor_ops as TO
    x = torch.randn(10, 151, device=dev())
    with pytest.raises(_lib.PdpError):
        TO.TensorLinear(torch.nn.Linear(151, 257).to(dev()))([x])                          # > one accumulator block
    with pytest.raises(_lib.PdpError):
        TO.TensorLinear(torch.nn.Linear(1025, 4).to(dev()))([torch.randn(10, 1025, device=dev())])   # > 64 K chunks


# ---------------------------------------------------------------------------------------------------------------------
# GRU cell
# ---------------------------------------------------------------------------------------------------------------------
def _gru_case(rows, pieces, H, mask="binary", x_offset=(), h_offset=False, seed=0):
    from pdp_solver_b200.nn import tensor_ops as TO
    kx = sum(pieces)
    torch.manual_seed(seed)
    cell = torch.nn.GRUCell(kx, H).to(dev())
    w_ih, w_hh, b_ih, b_hh = (C(p) for p in (cell.weight_ih, cell.weight_hh, cell.bias_ih, cell.bias_hh))
    rng = np.random.default_rng(seed)
    xh = NR.coherent_rows(rng.uniform(-1, 1, (rows, H + kx)).astype(np.float32), np.concatenate((w_hh, w_ih), 1)[2 * H:], -0.25)
    h, x = np.ascontiguousarray(xh[:, :H]), xh[:, H:]
    cuts = np.cumsum([0] + list(pieces))
    src = [on_device(x[:, cuts[i]:cuts[i + 1]], i in x_offset) for i in range(len(pieces))]
    hd = on_device(h, h_offset)
    m = {"none": None, "binary": (rng.random(rows) > 0.2).astype(np.float32)}[mask]
    out = TO.TensorGRU(cell)(src, hd, row_mask=None if m is None else on_device(m))
    ref, tol = NR.gru64(x, h, w_ih, w_hh, b_ih, b_hh, m)
    got = C(out).astype(np.float64)
    assert (np.abs(got - ref) <= tol).all(), "max error/tol %.2f" % _note("gru", got - ref, tol)
    _note("gru", got - ref, tol)
    if m is not None:
        assert np.array_equal(C(out)[m == 0].view(np.int32), h[m == 0].view(np.int32))     # frozen rows: h bit for bit
    return cell, src, hd, out


# (rows, x pieces, H, mask, x offsets, h offset)
GRU_CASES = (
    # H: one pass (61: last group of four units partial), 76: one pass of 304 columns -- the two accumulator buffers share
    # 96 columns, >= 3 tiles per CTA so the overlap barrier changes phase across tiles; 77, 150: two passes (150 overlaps);
    # 153, 192: three passes
    [("h%d" % H, (1001 if H != 76 else "3sms128+17", (150, 1), H, "binary", (), False)) for H in NR.GRU_H] +
    [("kx%d" % kx, (1001, (kx,), 150, "binary", (), False)) for kx in NR.GRU_KX] +
    [
        ("kx2_two_pieces", (1001, (1, 1), 150, "none", (), False)),
        ("kx3_two_pieces", (1001, (2, 1), 150, "binary", (), False)),
        ("h150_3tiles_per_cta", ("3sms128+17", (150, 1), 150, "binary", (), False)),
        ("x_offset", (1001, (150, 1), 150, "binary", (0,), False)),
        ("h_offset_vector_epilogue_falls_back", (1001, (150, 1), 150, "binary", (), True)),
        ("h_offset_h76_one_wide_pass", (1001, (150, 1), 76, "none", (), True)),
        ("h_and_x_offset_h4", (1001, (150, 1), 4, "binary", (0,), True)),
    ]
)


@pytest.mark.parametrize("case", [c for _, c in GRU_CASES], ids=[i for i, _ in GRU_CASES])
def test_gru_vs_fp64(case):
    rows, pieces, H, mask, x_offset, h_offset = case
    _gru_case(rows_of(rows), pieces, H, mask, x_offset, h_offset, seed=H + sum(pieces))


def test_gru_rejects_what_does_not_fit():
    from pdp_solver_b200 import _lib
    from pdp_solver_b200.nn import tensor_ops as TO
    with pytest.raises(_lib.PdpError):      # 193 units: three passes of 272 columns > the 768 bias columns
        TO.TensorGRU(torch.nn.GRUCell(3, 193).to(dev()))([torch.randn(10, 3, device=dev())], torch.zeros(10, 193, device=dev()))
    # out aliasing h is refused by the C entry point
    cell = torch.nn.GRUCell(3, 8).to(dev())
    g = TO.TensorGRU(cell)
    g([torch.randn(4, 3, device=dev())], torch.zeros(4, 8, device=dev()))
    L = _lib.load()
    x, h = torch.randn(4, 3, device=dev()), torch.zeros(4, 8, device=dev())
    p = lambda t: ctypes.c_void_p(t.data_ptr())
    rc = L.pdp_edge_gru_forward(p(x), 3, ctypes.c_void_p(0), 0, p(h), 8, 4, p(g.image), p(g.bias), g.n_blk, g.n_mma, g.passes,
                                ctypes.c_void_p(0), p(h), ctypes.c_void_p(torch.cuda.current_stream().cuda_stream))
    assert rc != 0


# ---------------------------------------------------------------------------------------------------------------------
# bitwise invariances
# ---------------------------------------------------------------------------------------------------------------------
def test_row_independence_bitwise():
    """a row's result depends on that row only: permuting or truncating the rows permutes or truncates the results,
    bit for bit (no cross-row state in the tile pipeline, whatever tile or CTA a row lands in)"""
    from pdp_solver_b200.nn import tensor_ops as TO
    n = rows_of("sms128+1")
    perm = torch.randperm(n, generator=torch.Generator().manual_seed(3)).to(dev())
    lin, src, out = _linear_case(n, (150, 1), 100, 1, "fraction", seed=11)
    t = TO.TensorLinear(lin)
    assert torch.equal(t([s[perm] for s in src], act=1), t(src, act=1)[perm])
    assert torch.equal(t([s[:777] for s in src], act=1), t(src, act=1)[:777])
    cell, xs, h, _ = _gru_case(n, (150, 1), 150, "none", seed=12)
    g = TO.TensorGRU(cell)
    full = g(xs, h)
    assert torch.equal(g([s[perm] for s in xs], h[perm]), full[perm])
    assert torch.equal(g([s[:777] for s in xs], h[:777]), full[:777])


def test_ring_depth_and_store_path_bitwise(monkeypatch):
    """PDP_B200_NN_STAGES = 2, 3, 4 (shared-memory stages of the operand ring; a depth that does not fit beside the copy
    ring is ignored: the GRU cell's 304-column stages take at most 3) and PDP_B200_NN_OTILE = 0 (thread-per-row stores
    instead of the tile's bulk store) change the schedule only: identical bytes"""
    from pdp_solver_b200.nn import tensor_ops as TO
    n = rows_of("3sms128+17")
    lin, src, _ = _linear_case(n, (150, 1), 100, 1, "none", seed=21)
    cell, xs, h, _ = _gru_case(n, (150, 1), 150, "binary", seed=22)
    mk = torch.from_numpy((np.arange(n) % 5 != 0).astype(np.float32)).to(dev())
    ref_l = TO.TensorLinear(lin)(src, act=1, row_mask=mk)
    ref_g = TO.TensorGRU(cell)(xs, h, row_mask=mk)
    for st in ("2", "3", "4"):
        monkeypatch.setenv("PDP_B200_NN_STAGES", st)
        assert torch.equal(TO.TensorLinear(lin)(src, act=1, row_mask=mk), ref_l), "stages " + st
        assert torch.equal(TO.TensorGRU(cell)(xs, h, row_mask=mk), ref_g), "stages " + st
        monkeypatch.setenv("PDP_B200_NN_OTILE", "0")
        assert torch.equal(TO.TensorLinear(lin)(src, act=1, row_mask=mk), ref_l), "thread-per-row stores, stages " + st
        monkeypatch.delenv("PDP_B200_NN_OTILE")


# ---------------------------------------------------------------------------------------------------------------------
# pdp_edge_aggregate
# ---------------------------------------------------------------------------------------------------------------------
@pytest.fixture(scope="module")
def agg_graph():
    """one problem, 3 literals per clause, edges in a random order; variable 0 on 4 500 edges, the last 10 variables on
    none; V = 100 000: the warp-per-node loop wraps several times at every channel count"""
    from pdp_solver_b200.engine import Context
    rng = np.random.default_rng(5)
    V, F = 100000, 110000
    E = 3 * F
    var = rng.integers(1, V - 10, E).astype(np.int32)
    var[rng.choice(E, 4500, replace=False)] = 0
    cls = (np.arange(E) // 3).astype(np.int32)
    perm = rng.permutation(E)
    gm = np.ascontiguousarray(np.stack((var, cls))[:, perm])
    ef = np.where(rng.random(E) < 0.5, -1.0, 1.0).astype(np.float32)
    bvm, bfm = np.zeros(V, np.int32), np.zeros(F, np.int32)
    ctx = Context(*(torch.from_numpy(a).to(dev()) for a in (gm, bvm, bfm, ef)))
    return ctx, gm, V, F


@pytest.mark.parametrize("C_", [1, 2, 31, 32, 33, 50, 64, 100, 150])
@pytest.mark.parametrize("by_variable", [True, False], ids=["by_variable", "by_clause"])
def test_edge_aggregate_bitwise_sequential_fp32(agg_graph, C_, by_variable):
    ctx, gm, V, F = agg_graph
    E = gm.shape[1]
    nodes, node_of_edge = (V, gm[0]) if by_variable else (F, gm[1])
    rng = np.random.default_rng(C_)
    # magnitudes over 12 decades: a different summation order rounds differently
    state = (rng.standard_normal((E, C_)) * 10.0 ** rng.integers(-6, 7, (E, C_))).astype(np.float32)
    loo_on = C_ % 2 == 1 or C_ == 150
    s, loo = ctx.edge_aggregate(torch.from_numpy(state).to(dev()), by_variable=by_variable, leave_one_out=loo_on)
    seq, seq_loo = NR.segment_sum_seq32(state, node_of_edge, nodes)
    got = C(s)
    assert np.array_equal(got.view(np.int32), seq.view(np.int32))
    if by_variable:
        assert (got[-10:] == 0).all() and np.bincount(gm[0], minlength=V)[0] >= 4000
    s64, mag = NR.segment_sum64(state, node_of_edge, nodes)
    deg = np.bincount(node_of_edge, minlength=nodes).astype(np.float64)[:, None]
    tol = deg * NR.U24 * mag + 1e-45
    assert (np.abs(got - s64) <= tol).all()
    _note("edge_aggregate", got - s64, tol)
    if loo_on:
        gl = C(loo)
        assert np.array_equal(gl.view(np.int32), seq_loo.view(np.int32))
        ref = s64[node_of_edge] - state
        ltol = tol[node_of_edge] + NR.U24 * np.abs(ref) + 1e-45
        assert (np.abs(gl - ref) <= ltol).all()
    else:
        assert loo is None


# ---------------------------------------------------------------------------------------------------------------------
# SP step on adaptor outputs; pdp_sp_step / pdp_score at pi != 0
# ---------------------------------------------------------------------------------------------------------------------
@pytest.fixture(scope="module")
def sp_batch():
    from pdp_solver_b200 import cnfgen
    gm, bvm, bfm, ef = cnfgen.mixed_batch([(3000, 3, 4.2), (500, 4, 9.0), (2000, 3, 3.8), (40, 2, 1.0), (1000, 5, 20.0)], 17)
    perm = np.random.default_rng(17).permutation(gm.shape[1])
    return np.ascontiguousarray(gm[:, perm]), bvm, bfm, np.ascontiguousarray(ef[perm])


def _sp_inputs(E, B, seed):
    rng = np.random.default_rng(seed)
    q = rng.random((E, 3)).astype(np.float32)
    q[rng.random(E) < 0.02, 0] = 0.0                       # log(max(0, 1e-40)): the clamp
    q /= np.maximum(q.sum(1, keepdims=True), 1e-30).astype(np.float32)
    df = np.stack((rng.random(E), np.sign(rng.standard_normal(E))), 1).astype(np.float32)
    pq, pf = rng.random((E, 3)).astype(np.float32), rng.random((E, 2)).astype(np.float32)
    em = (rng.random(E) > 0.25).astype(np.float32)
    active = (rng.random(B) > 0.3).astype(np.uint8)
    active[0], active[1] = 1, 0
    return q, df, pq, pf, em, active


@pytest.mark.parametrize("pi", [0.0, 0.1, 0.5])
def test_sp_step_adapted(sp_batch, pi):
    from pdp_solver_b200.engine import Context
    gm, bvm, bfm, ef = sp_batch
    E, V, F, B = gm.shape[1], bvm.shape[0], bfm.shape[0], int(bvm.max()) + 1
    q, df, pq, pf, em, active = _sp_inputs(E, B, int(pi * 10) + 1)
    T = lambda a: torch.from_numpy(np.ascontiguousarray(a)).to(dev())
    # strict-math build: x_log = the build's own L40 of q (correctly rounded log of max(q, 1e-40f)) -> bit for bit sp_step
    x_log = np.log(np.maximum(q[:, 0], np.float32(1e-40)).astype(np.float64)).astype(np.float32)
    ctx = Context(T(gm), T(bvm), T(bfm), T(ef), strict_math=True)
    a_q, a_f = ctx.sp_step_adapted(T(x_log), T(df[:, 0]), T(df[:, 1]), T(em), T(pq), T(pf), T(active), pi)
    b_q, b_f = ctx.sp_step(T(q), T(df), T(em), T(pq), T(pf), T(active), pi)
    assert torch.equal(a_q, b_q) and torch.equal(a_f, b_f)
    # product build against the float64 restatement
    ctx = Context(T(gm), T(bvm), T(bfm), T(ef))
    gq, gf = ctx.sp_step_adapted(T(x_log), T(df[:, 0]), T(df[:, 1]), T(em), T(pq), T(pf), T(active), pi)
    rq, rf, tq, tf = NR.sp_step64(gm, ef, bvm[gm[0]], V, F, x_log, df[:, 0], df[:, 1], em, pq, pf, active, pi)
    gq, gf = C(gq).astype(np.float64), C(gf).astype(np.float64)
    assert (np.abs(gq - rq) <= tq).all(), _note("sp_step_adapted", gq - rq, tq)
    assert (np.abs(gf - rf) <= tf).all(), _note("sp_step_adapted", gf - rf, np.maximum(tf, 1e-300))
    _note("sp_step_adapted", gq - rq, tq)
    _note("sp_step_adapted", (gf - rf)[:, 0][tf[:, 0] > 0], tf[:, 0][tf[:, 0] > 0])
    frozen = active[bvm[gm[0]]] == 0
    assert np.array_equal(gq[frozen], pq[frozen]) and np.array_equal(gf[frozen, 0], pf[frozen, 0])


@pytest.mark.parametrize("pi", [0.1, 0.5])
def test_sp_step_and_score_at_nonzero_pi_vs_oracle(sp_batch, pi):
    """pdp_sp_step and pdp_score with the external-force term (the goldens have pi = 0 only) against the C oracle"""
    from oracle import pdp_oracle as po
    from pdp_solver_b200.engine import Context
    gm, bvm, bfm, ef = sp_batch
    E, B = gm.shape[1], int(bvm.max()) + 1
    q, df, pq, pf, em, active = _sp_inputs(E, B, int(pi * 10) + 7)
    T = lambda a: torch.from_numpy(np.ascontiguousarray(a)).to(dev())
    ctx = Context(T(gm), T(bvm), T(bfm), T(ef))
    o = po.Oracle(gm, bvm, bfm, ef)
    gq, gf = ctx.sp_step(T(q), T(df), T(em), T(pq), T(pf), T(active), pi)
    gq, gf = C(gq), C(gf)
    oq, of = o.sp_step(q, df, em, pq, pf, active, pi)
    # a clause with a clamped message (log 1e-40 = -92.1) leaves tot - v with an absolute fp32 error of ~ulp(92): the
    # device and the oracle are each within the float64 bound, not within a fixed 2e-6 of each other
    x_log = np.log(np.maximum(q[:, 0], np.float32(1e-40)).astype(np.float64))
    rq, rf, tq, tf = NR.sp_step64(gm, ef, bvm[gm[0]], bvm.shape[0], bfm.shape[0], x_log, df[:, 0], df[:, 1], em, pq, pf, active, pi)
    for name, g, o_, r, tol in (("q", gq, oq, rq, tq), ("fs", gf, of, rf, tf)):
        for who, v in (("device", g), ("oracle", o_)):
            bad = ~(np.abs(v - r) <= tol)
            assert not bad.any(), "%s %s: %d outside, first at %s: %r, float64 %r" % (
                who, name, bad.sum(), np.argwhere(bad)[0], v[bad][:4].tolist(), r[bad][:4].tolist())
        _note("sp_step", g - r, np.maximum(tol, 1e-300))
    # the scorer's tail takes differences of exponentials (q0 = e^pos - e^(pos + neg)): a 1-ulp difference between the
    # device's and the C library's logf / expf can come out several ulps of 1 larger
    af = (np.random.default_rng(3).random(bfm.shape[0]) > 0.1).astype(np.float32)
    assert np.abs(C(ctx.score(T(df), T(af), pi)) - o.score(df, af, pi)).max() < 1e-5


# ---------------------------------------------------------------------------------------------------------------------
# whole models at the reference's dimensions (config/Predict/np-nd-np.yaml)
# ---------------------------------------------------------------------------------------------------------------------
H, MH, AH, MAH, CH = 150, 100, 100, 50, 50


def _model(kind):
    from pdp_solver_b200.nn import solver as S
    from pdp_solver_b200.nn import util as U
    common = dict(edge_dimension=1, meta_data_dimension=0, mem_hidden_dimension=MH, agg_hidden_dimension=AH,
                  mem_agg_hidden_dimension=MAH, local_search_iterations=0, epsilon=0.5)
    torch.manual_seed(1234)
    if kind == "p-nd-np":
        return S.NeuralSurveyPropagatorSolver(dev(), "m", decimator_dimension=H, prediction_dimension=1,
                                              variable_classifier=U.Perceptron(H, CH, 1), function_classifier=None, dropout=0, **common)
    if kind == "np-nd-np":
        return S.NeuralPropagatorDecimatorSolver(dev(), "m", propagator_dimension=H, decimator_dimension=H, prediction_dimension=1,
                                                 variable_classifier=U.Perceptron(H, CH, 1), function_classifier=None, dropout=0, **common)
    return S.NeuralSequentialDecimatorSolver(dev(), "m", propagator_dimension=H, decimator_dimension=H, classifier_dimension=CH,
                                             dropout=0, tolerance=0.02, t_max=100, **common)


def _layer_bound(model):
    """the largest per-output bound of any dense layer of the model for inputs of size <= 1:
    C_GEMM (K 2^-24 + 2^-20) max_n sum_k |w_nk| -- the GRU cells' input and hidden weights side by side"""
    worst = 0.0
    for m in model.modules():
        if isinstance(m, torch.nn.Linear):
            w = m.weight.detach().abs()
        elif isinstance(m, torch.nn.GRUCell):
            w = torch.cat((m.weight_ih, m.weight_hh), 1).detach().abs()
        else:
            continue
        worst = max(worst, NR.C_GEMM * (w.shape[1] * NR.U24 + 2.0 ** -20) * float(w.sum(1).max()))
    return worst


@pytest.mark.parametrize("kind", ["p-nd-np", "np-nd-np", "np-d-np"])
def test_whole_model_tcgen05_vs_library_gemm(kind, monkeypatch):
    """forward() with the dense layers on tcgen05 against the same model on fp32 library GEMMs (tf32 off): agreement
    within the per-layer bound, times the layers a value passes through per iteration (<= 8) and the iterations"""
    from pdp_solver_b200 import cnfgen
    iters = 2
    batch = cnfgen.random_batch(4, 1200, 3, 4.2, 99)
    E = batch[0].shape[1]
    assert E >= 3 * sms() * 128
    gm, bvm, bfm, ef = (torch.from_numpy(np.ascontiguousarray(a)).to(dev()) for a in batch)
    base = _model(kind).to(dev()).eval()
    sd = base.state_dict()
    bound = _layer_bound(base)
    torch.manual_seed(7)
    init = base.get_init_state(gm, bvm, bfm, ef, None, randomized=True, batch_replication=1)

    def termination(active, prediction, sat_problem):
        raise RuntimeError("unreachable")
    termination._pdp_standard_termination = True
    monkeypatch.setattr(torch.backends.cuda.matmul, "allow_tf32", False)
    outs = []
    for mode in ("tcgen05", "torch"):
        monkeypatch.setenv("PDP_B200_NN", mode)
        model = _model(kind).to(dev()).eval()
        model.load_state_dict(sd)
        if kind == "np-d-np":
            model.get_init_state(gm, bvm, bfm, ef, None, randomized=False, batch_replication=1)    # resets the decimator
        st = tuple(None if part is None else tuple(t.clone() for t in part) for part in init)
        with torch.no_grad():
            (vp, _), (ps, ds) = model(init_state=st, graph_map=gm, batch_variable_map=bvm, batch_function_map=bfm, edge_feature=ef,
                                      meta_data=None, is_training=False, iteration_num=iters,
                                      check_termination=None if kind == "np-d-np" else termination, simplify=True, batch_replication=1)
        outs.append([C(t).astype(np.float64) for t in (vp,) + tuple(ps) + tuple(ds) if torch.is_tensor(t)])
    tol = 8 * iters * bound + NR.C_SFU
    for a, b in zip(*outs):
        err = np.abs(a - b)
        assert (err <= tol).all(), "max |difference| %.3g, tolerance %.3g" % (err.max(), tol)
        _note("whole_model", err, tol)
