"""CPU checks of the float64 restatements in tests/neural_reference.py: that they compute what the library's operators are
specified to compute, and that the tf32 error bound is tight enough to catch a kernel that loses a split term."""
import numpy as np
import pytest
import torch

from tests import neural_reference as NR


def test_gru64_equals_torch_grucell_in_float64():
    torch.manual_seed(0)
    for kx, H, bias in ((151, 150, True), (3, 7, False), (1, 1, True)):
        cell = torch.nn.GRUCell(kx, H, bias=bias).double()
        x, h = torch.randn(37, kx, dtype=torch.float64), torch.rand(37, H, dtype=torch.float64) * 2 - 1
        with torch.no_grad():
            ref = cell(x, h).numpy()
        b = (cell.bias_ih.detach().numpy(), cell.bias_hh.detach().numpy()) if bias else (None, None)
        got, tol = NR.gru64(x.numpy(), h.numpy(), cell.weight_ih.detach().numpy(), cell.weight_hh.detach().numpy(), *b)
        assert np.abs(got - ref).max() < 1e-13
        assert (tol > 0).all()
        # the frozen-row blend: rows whose mask is 0 keep h exactly
        mask = (np.arange(37) % 3 != 0).astype(np.float64)
        got_m, _ = NR.gru64(x.numpy(), h.numpy(), cell.weight_ih.detach().numpy(), cell.weight_hh.detach().numpy(), *b, row_mask=mask)
        assert np.array_equal(got_m[mask == 0], h.numpy()[mask == 0])
        assert np.array_equal(got_m[mask == 1], got[mask == 1])


def test_linear64_equals_torch_linear_in_float64():
    torch.manual_seed(1)
    lin = torch.nn.Linear(151, 100).double()
    x = torch.randn(50, 151, dtype=torch.float64)
    mask = torch.rand(50, dtype=torch.float64)
    with torch.no_grad():
        ref = (torch.nn.functional.logsigmoid(lin(x)) * mask[:, None]).numpy()
    got, _ = NR.linear64(x.numpy(), lin.weight.detach().numpy(), lin.bias.detach().numpy(), act=1, row_mask=mask.numpy())
    assert np.abs(got - ref).max() < 1e-13


def test_tf32_split_matches_the_host_side_split():
    from pdp_solver_b200.nn import tensor_ops
    x = torch.randn(1000) * torch.logspace(-20, 20, 1000)
    hi, lo = tensor_ops._tf32_split(x)
    nhi, nlo = NR.tf32_split(x.numpy())
    assert np.array_equal(hi.numpy().view(np.int32), nhi.view(np.int32)) and np.array_equal(lo.numpy().view(np.int32), nlo.view(np.int32))
    # hi keeps 10 explicit mantissa bits, lo the next 11: what is left is below 2^-21 of x
    r = x.numpy().astype(np.float64) - nhi - nlo
    assert (np.abs(r) <= 2.0 ** -21 * np.abs(x.numpy())).all()


def _seq_loop(state, node_of_edge, nodes):
    out = np.zeros((nodes, state.shape[1]), np.float32)
    for ch in range(state.shape[1]):
        for i in range(nodes):
            acc = np.float32(0.0)
            for e in range(state.shape[0]):          # ascending edge index
                if node_of_edge[e] == i:
                    acc = np.float32(acc + state[e, ch])
            out[i, ch] = acc
    return out


def test_sequential_fp32_sum_equals_a_python_loop():
    rng = np.random.default_rng(2)
    E, nodes, C = 400, 37, 3
    node_of_edge = rng.integers(0, nodes - 2, E)          # the last two nodes have no edge
    # values of very different sizes: any other summation order would round differently
    state = (rng.standard_normal((E, C)) * 10.0 ** rng.integers(-6, 7, (E, C))).astype(np.float32)
    got, loo = NR.segment_sum_seq32(state, node_of_edge, nodes)
    ref = _seq_loop(state, node_of_edge, nodes)
    assert np.array_equal(got.view(np.int32), ref.view(np.int32))
    assert (got[-2:] == 0).all()
    assert np.array_equal(loo, (ref[node_of_edge] - state).astype(np.float32))
    s64, mag = NR.segment_sum64(state, node_of_edge, nodes)
    assert (np.abs(got - s64) <= E * NR.U24 * mag).all()


def _rows(rng, n, k, w):
    x = rng.standard_normal((n, k)).astype(np.float32)
    return NR.coherent_rows(x, w, -8.0)


@pytest.mark.parametrize("shape", NR.linear_shapes(), ids=lambda s: "K%d_n%d" % s)
def test_linear_bound_sensitivity(shape):
    """the three-term emulation stays inside the bound; the emulations without the lo*hi or the hi*lo products leave it"""
    K, n = shape
    rng = np.random.default_rng(K * 1000 + n)
    w = (rng.uniform(-1, 1, (n, K)) / np.sqrt(K)).astype(np.float32)
    x = _rows(rng, 64, K, w)
    for act in (0, 1):
        ref, tol = NR.linear64(x, w, act=act)
        f = (lambda y: NR.logsigmoid64(y)) if act else (lambda y: y)
        full = f(NR.gemm_split64(x, w))
        assert (np.abs(full - ref) <= tol).all()
        for drop in ("lh", "hl"):
            part = f(NR.gemm_split64(x, w, tuple(t for t in ("hh", "lh", "hl") if t != drop)))
            assert (np.abs(part - ref) > tol).any(), "a kernel without the %s products would pass" % drop


@pytest.mark.parametrize("shape", NR.gru_shapes(), ids=lambda s: "kx%d_h%d" % s)
def test_gru_bound_sensitivity(shape):
    kx, H = shape
    rng = np.random.default_rng(kx * 1000 + H)
    s = 1 / np.sqrt(H)
    w_ih = rng.uniform(-s, s, (3 * H, kx)).astype(np.float32)
    w_hh = rng.uniform(-s, s, (3 * H, H)).astype(np.float32)
    b_ih, b_hh = (rng.uniform(-s, s, 3 * H).astype(np.float32) for _ in range(2))
    w_all = np.concatenate((w_hh, w_ih), 1)
    xh = NR.coherent_rows(rng.uniform(-1, 1, (64, H + kx)).astype(np.float32), w_all[2 * H:], -0.25)
    h, x = xh[:, :H], xh[:, H:]
    ref, tol = NR.gru64(x, h, w_ih, w_hh, b_ih, b_hh)
    full, _ = NR.gru64(x, h, w_ih, w_hh, b_ih, b_hh, terms=("hh", "lh", "hl"))
    assert (np.abs(full - ref) <= tol).all()
    for drop in ("lh", "hl"):
        part, _ = NR.gru64(x, h, w_ih, w_hh, b_ih, b_hh, terms=tuple(t for t in ("hh", "lh", "hl") if t != drop))
        assert (np.abs(part - ref) > tol).any(), "a kernel without the %s products would pass" % drop


@pytest.mark.parametrize("pi", [0.0, 0.1, 0.5])
def test_sp_step64_equals_the_c_oracle(pi):
    """the float64 SP step on adaptor inputs, fed log(q) and the decimator's surveys, against the C oracle's pdp_sp_step
    (which takes log(max(q, 1e-40)) itself): random edge masks, some problems inactive, a permuted edge order"""
    from oracle import pdp_oracle as po
    from pdp_solver_b200 import cnfgen
    gm, bvm, bfm, ef = cnfgen.mixed_batch([(40, 3, 4.0), (25, 4, 8.0), (60, 3, 3.5), (10, 2, 1.0)], 7)
    E = gm.shape[1]
    rng = np.random.default_rng(int(pi * 10))
    perm = rng.permutation(E)
    gm, ef = np.ascontiguousarray(gm[:, perm]), np.ascontiguousarray(ef[perm])
    V, F, B = bvm.shape[0], bfm.shape[0], int(bvm.max()) + 1
    q = rng.random((E, 3)).astype(np.float32)
    q /= q.sum(1, keepdims=True)
    df = np.stack((rng.random(E), np.sign(rng.standard_normal(E))), 1).astype(np.float32)
    pq, pf = rng.random((E, 3)).astype(np.float32), rng.random((E, 2)).astype(np.float32)
    em = (rng.random(E) > 0.25).astype(np.float32)
    active = np.array([1, 0, 1, 1], np.uint8)[:B]
    o = po.Oracle(gm, bvm, bfm, ef)
    oq, of = o.sp_step(q, df, em, pq, pf, active, pi)
    x_log = np.log(np.maximum(q[:, 0].astype(np.float64), 1e-40))
    rq, rf, tq, tf = NR.sp_step64(gm, ef, bvm[gm[0]], V, F, x_log, df[:, 0], df[:, 1], em, pq, pf, active, pi)
    assert (np.abs(oq - rq) <= tq).all()
    assert (np.abs(of - rf) <= tf).all()
    frozen = active[bvm[gm[0]]] == 0
    assert frozen.any() and np.array_equal(oq[frozen], pq[frozen]) and np.array_equal(of[frozen, 0], pf[frozen, 0])
