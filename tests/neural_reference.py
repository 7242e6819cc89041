"""Plain float64 restatements of the device operators of the neural model types (no GPU needed):

- the dense layer and torch.nn.GRUCell (with the frozen-row blend) of pdp_edge_mlp_forward / pdp_edge_gru_forward,
  an elementwise error bound for their three-term tf32 split, and a float64 emulation of that split;
- the segmented sums of pdp_edge_aggregate, in float64 and in sequential float32 (ascending edge order);
- the SP step on adaptor outputs of pdp_sp_step_adapted (reference pdp_propagate.py:139-221).

Everything works on numpy arrays; the callers move tensors to the host first."""
import numpy as np

# ---------------------------------------------------------------------------------------------------------------------
# dense layer, GRU cell
# ---------------------------------------------------------------------------------------------------------------------
U24 = 2.0 ** -24
# Error bound of one output of the tf32 three-term product A W^T (csrc/pdp_edge_nn.cu):
#   |got - exact| <= C_GEMM * (K * 2^-24 + 2^-20) * sum_k |a_k| |w_k|
# - the split: x = hi + lo + r with |lo| < 2^-10 |x| and |r| < 2^-21 |x| (both parts truncated to 19 bits); the three
#   products kept leave lo_a lo_w + r_a w + hi_a r_w, at most (2^-20 + 2 * 2^-21) |a||w| = 2 * 2^-20 |a||w|;
# - fp32 accumulation in tensor memory of the 3K products: the tensor core adds with truncation (no guard bits), a
#   relative error up to 2^-23 per addition.  Worst case 3K * 2^-23 = 6K * 2^-24, but that needs every partial sum at
#   full size; with the partial sums growing from 0 the expected truncation error of a one-signed row is about half an
#   ulp per addition of the products that matter (hi hi) plus the small lo terms: ~1.5 K * 2^-24.
# C_GEMM = 4 keeps a factor 2 over the split's residual and ~2.7 over that accumulation estimate, and stays below the
# size of one dropped split term (~2^-11.5 sum |a||w| on rows whose products share a sign) up to K = 1024: a kernel that
# lost the lo*hi or the hi*lo products fails the bound (test_neural_reference.py checks both directions on the CPU).
C_GEMM = 4.0
# Epilogue on the special-function unit: __expf / __logf / __fdividef have relative (for __logf absolute, on [0.5, 2])
# errors of ~2^-21; logsigmoid and sigmoid add one or two of them and a few fp32 roundings of O(|ref|) values.  The GRU
# cell chains two sigmoids and a tanh (2 sigmoid(2x) - 1).  C_SFU = 2^-18 (8x the SFU error) covers them all.
C_SFU = 2.0 ** -18


def tf32_split(x):
    """(hi, lo) of the kernel's split: hi = x truncated to 19 bits (tf32), lo = (x - hi) truncated the same way -- the rule of
    tensor_ops._tf32_split, for the weights and for the operand rows alike"""
    x = np.ascontiguousarray(x, dtype=np.float32)
    hi = (x.view(np.int32) & np.int32(-8192)).view(np.float32)
    d = np.ascontiguousarray(x - hi, dtype=np.float32)
    lo = (d.view(np.int32) & np.int32(-8192)).view(np.float32)
    return hi, lo


def gemm64(a, w):
    "A W^T in float64"
    return np.asarray(a, np.float64) @ np.asarray(w, np.float64).T


def gemm_split64(a, w, terms=("hh", "lh", "hl")):
    """A W^T as the kernel forms it -- the sum of the split products named in `terms` (first letter: A's part, second:
    W's) -- with the products and the sum in float64: only the split is emulated, not the fp32 accumulation"""
    ah, al = tf32_split(a)
    wh, wl = tf32_split(w)
    parts = {"h": (ah, wh), "l": (al, wl)}
    out = np.zeros((np.shape(a)[0], np.shape(w)[0]))
    for t in terms:
        out += gemm64(parts[t[0]][0], parts[t[1]][1])
    return out


def gemm_bound(a, w):
    "the elementwise bound of the split product above (without the epilogue term)"
    k = np.shape(a)[1]
    return C_GEMM * (k * U24 + 2.0 ** -20) * (np.abs(np.asarray(a, np.float64)) @ np.abs(np.asarray(w, np.float64)).T)


def logsigmoid64(x):
    return np.minimum(x, 0.0) - np.log1p(np.exp(-np.abs(x)))


def sigmoid64(x):
    return 0.5 * (1.0 + np.tanh(0.5 * x))


def linear64(a, w, b=None, act=0, row_mask=None):
    """act([a] W^T + b) * row_mask in float64 and its elementwise tolerance.  logsigmoid is 1-Lipschitz: the product's
    bound passes through it unchanged."""
    y = gemm64(a, w)
    if b is not None:
        y = y + np.asarray(b, np.float64)
    if act:
        y = logsigmoid64(y)
    tol = gemm_bound(a, w)
    if row_mask is not None:
        m = np.asarray(row_mask, np.float64).reshape(-1, 1)
        y, tol = y * m, tol * np.abs(m)
    return y, tol + C_SFU * (1.0 + np.abs(y))


def gru64(x, h, w_ih, w_hh, b_ih=None, b_hh=None, row_mask=None, terms=None):
    """torch.nn.GRUCell in float64, written out:
        r = sigmoid(W_ir x + b_ir + W_hr h + b_hr),  z = sigmoid(W_iz x + b_iz + W_hz h + b_hz)
        n = tanh(W_in x + b_in + r * (W_hn h + b_hn)),  h' = (1 - z) * n + z * h
    then h' blended with h where row_mask is 0 (mask * h' + (1 - mask) * h).  Returns (h', tol).  The tolerance carries
    each pre-activation's product bound through the gates: sigmoid is 1/4-Lipschitz, tanh 1-Lipschitz, so
        |dh'| <= (1 - z) (e_in + r e_hn + |W_hn h + b_hn| e_r / 4) + |h - n| e_z / 4.
    With `terms` the products take the split emulation (gemm_split64) instead of the exact float64 ones."""
    x, h = np.asarray(x, np.float64), np.asarray(h, np.float64)
    H = h.shape[1]
    mm = gemm64 if terms is None else (lambda a, w: gemm_split64(a, w, terms))
    # the kernel's rows are [h | x]; every gate column is one product over that row (r and z: both parts together)
    xh = np.concatenate((h, x), 1)
    w_all = np.concatenate((w_hh, w_ih), 1)       # [3H, H + kx]
    gi = mm(x, w_ih)
    gh = mm(h, w_hh)
    rz = mm(xh, w_all[:2 * H])
    b_ih = np.zeros(3 * H) if b_ih is None else np.asarray(b_ih, np.float64)
    b_hh = np.zeros(3 * H) if b_hh is None else np.asarray(b_hh, np.float64)
    r = sigmoid64(rz[:, :H] + b_ih[:H] + b_hh[:H])
    z = sigmoid64(rz[:, H:] + b_ih[H:2 * H] + b_hh[H:2 * H])
    hn = gh[:, 2 * H:] + b_hh[2 * H:]
    n = np.tanh(gi[:, 2 * H:] + b_ih[2 * H:] + r * hn)
    out = (1.0 - z) * n + z * h
    e_rz = gemm_bound(xh, w_all[:2 * H])
    e_in = gemm_bound(x, np.asarray(w_ih)[2 * H:])
    e_hn = gemm_bound(h, np.asarray(w_hh)[2 * H:])
    tol = (1.0 - z) * (e_in + r * e_hn + np.abs(hn) * e_rz[:, :H] / 4) + np.abs(h - n) * e_rz[:, H:] / 4
    if row_mask is not None:
        m = np.asarray(row_mask, np.float64).reshape(-1, 1)
        out = m * out + (1.0 - m) * h
        tol = tol * np.abs(m)
    return out, tol + C_SFU * (1.0 + np.abs(out))


def coherent_rows(x, w, target, every=4):
    """x with every `every`-th row made one-signed against one weight row (row i: x[i, k] = -|x[i, k]| sign(w[i % N, k])):
    in those rows the products of one output share a sign, so a dropped split term adds up instead of averaging out.
    The row is scaled so that the sum is `target` (< 0): where the activation that follows has a slope near 1, not where
    it saturates (logsigmoid: well below 0; tanh: near 0)."""
    x = np.array(x, np.float32, copy=True)
    n = np.shape(w)[0]
    for i in range(0, x.shape[0], every):
        s = np.sign(np.asarray(w)[i % n, :x.shape[1]])
        s[s == 0] = 1
        x[i] = -np.abs(x[i]) * s
        x[i] *= np.float32(-target / (np.abs(x[i]) @ np.abs(np.asarray(w[i % n, :x.shape[1]], np.float32))))
    return x


# ---------------------------------------------------------------------------------------------------------------------
# segmented sums (MessageAggregator, reference util.py:51-77)
# ---------------------------------------------------------------------------------------------------------------------
def node_edges(node_of_edge, nodes):
    "(ptr, order): the edges of node i are order[ptr[i]:ptr[i + 1]], in ascending edge index"
    node_of_edge = np.asarray(node_of_edge, np.int64)
    order = np.argsort(node_of_edge, kind="stable")
    ptr = np.zeros(nodes + 1, np.int64)
    np.add.at(ptr, node_of_edge + 1, 1)
    return np.cumsum(ptr), order


def segment_sum64(state, node_of_edge, nodes):
    "node sums in float64, their bound sum |x| and the leave-one-out gather back to the edges"
    state = np.asarray(state, np.float64)
    out = np.zeros((nodes, state.shape[1]))
    mag = np.zeros_like(out)
    np.add.at(out, node_of_edge, state)
    np.add.at(mag, node_of_edge, np.abs(state))
    return out, mag


def segment_sum_seq32(state, node_of_edge, nodes):
    """node sums in float32, each node's edges added left to right in ascending edge index, and the leave-one-out
    fl(sum - x) of every edge.  The loop runs over the position inside a node, not over the nodes: step j adds the j-th
    edge of every node that has one, in float32 -- per node the same sequence of roundings as a left-to-right loop."""
    state = np.asarray(state, np.float32)
    ptr, order = node_edges(node_of_edge, nodes)
    deg = ptr[1:] - ptr[:-1]
    out = np.zeros((nodes, state.shape[1]), np.float32)
    for j in range(int(deg.max()) if nodes else 0):
        live = np.nonzero(deg > j)[0]
        out[live] = out[live] + state[order[ptr[live] + j]]
    loo = (out[np.asarray(node_of_edge)] - state).astype(np.float32)
    return out, loo


# ---------------------------------------------------------------------------------------------------------------------
# SP step on adaptor outputs (pdp_propagate.py:139-221; csrc/pdp_ops.cu k_sp_step_clause / k_sp_step_var)
# ---------------------------------------------------------------------------------------------------------------------
def _l40(x):
    "safe_log: log(max(x, 1e-40)) (pdp_propagate.py:133-134; NaN propagates)"
    return np.log(np.maximum(np.asarray(x, np.float64), 1e-40))


def _x30(x):
    "safe_exp: exp(min(x, 30))"
    return np.exp(np.minimum(x, 30.0))


def sp_step64(graph_map, edge_feature, problem_of_edge, V, F, x_log, eta_in, ext_in, edge_mask, prop_q3, prop_fs2,
              active=None, pi=0.0):
    """One SurveyPropagator.forward with the adaptors applied (x_log = logsigmoid of the function projector, eta_in =
    sigmoid and ext_in = sign of the variable projector), in float64.  Returns (q3 [E,3], fs2 [E,2], tol_q, tol_f): the
    tolerances bound what fp32 logarithms, exponentials and sums of the inputs can change (see sp_bounds)."""
    var, cls = np.asarray(graph_map[0], np.int64), np.asarray(graph_map[1], np.int64)
    E = var.shape[0]
    em = np.ones(E) if edge_mask is None else np.asarray(edge_mask, np.float64).reshape(-1)
    mask = np.ones(E) if active is None else np.asarray(active, np.float64).reshape(-1)[problem_of_edge]
    x_log, eta, ext = (np.asarray(t, np.float64).reshape(-1) for t in (x_log, eta_in, ext_in))
    pq, pf = np.asarray(prop_q3, np.float64), np.asarray(prop_fs2, np.float64)
    # clause side (:163-176): leave-one-out sum of the masked log messages of the clause
    v = x_log * em
    tot = np.zeros(F)
    np.add.at(tot, cls, v)
    fs = np.empty((E, 2))
    fs[:, 0] = np.where(mask != 0, mask * _x30(tot[cls] - v), pf[:, 0])
    fs[:, 1] = ext
    # variable side (:184-216): y = safe_log(1 - eta) * mask, split by the literal's sign
    y = _l40(1.0 - eta) * em
    neg = np.asarray(edge_feature).reshape(-1) < 0
    s = np.where(neg, -1.0, 1.0)
    P, N = np.zeros(V), np.zeros(V)
    np.add.at(P, var, np.where(neg, 0.0, y))
    np.add.at(N, var, np.where(neg, y, 0.0))
    Pe, Ne = P[var], N[var]
    same = 0.5 * (1 + s) * Pe + 0.5 * (1 - s) * Ne - y + _l40(1.0 - pi * (ext == s))
    opp = 0.5 * (1 - s) * Pe + 0.5 * (1 + s) * Ne + _l40(1.0 - pi * (ext == -s))
    S, O, dc = _x30(same), _x30(opp), _x30(same + opp)
    u, w = S * (1 - O), O * (1 - S)
    total = u + w + dc
    q = np.stack((u / total, w / total, dc / total), 1)
    q = np.where(mask[:, None] != 0, mask[:, None] * q, pq)
    # bounds: per node, the fp32 logarithms (~1 ulp each) and the fp32 sums of the degree's terms
    mag_c = np.zeros(F)
    np.add.at(mag_c, cls, np.abs(v))
    deg_c = np.bincount(cls, minlength=F).astype(np.float64)
    mag_v = np.zeros(V)
    np.add.at(mag_v, var, np.abs(y))
    deg_v = np.bincount(var, minlength=V).astype(np.float64)
    d_c = 4 * U24 * (deg_c[cls] + 2) * (mag_c[cls] + 1)        # absolute error of tot - v
    d_v = 4 * U24 * (deg_v[var] + 4) * (mag_v[var] + 2 - np.log1p(-pi))   # of same / opp
    tol_f = np.zeros((E, 2))
    # (+ two steps of the fp32 subnormal spacing 2^-149: a survey below 2^-126 keeps its absolute, not its relative error)
    tol_f[:, 0] = np.where(mask != 0, fs[:, 0] * (2 * d_c + 4 * U24) + 2.0 ** -148, 0.0)
    # q = (u, v, dc) / (S + O - S O) with S, O <= e^30: d q / d log S and d q / d log O are at most 2 in size (S, O <= 1)
    # and at most 2 max(S, O) / min-scale otherwise -- the inputs here keep the sums <= 0, so S, O, S O <= 1
    tol_q = np.where(mask[:, None] != 0, (4 * d_v)[:, None] + 16 * U24, 0.0) * np.ones((1, 3))
    return q, fs, tol_q, tol_f


# ---------------------------------------------------------------------------------------------------------------------
# the shapes the device tests run (tests/test_neural_ops_gpu.py); the CPU tests check the bound's sensitivity on each
# ---------------------------------------------------------------------------------------------------------------------
LINEAR_N_OUT = [1, 2, 15, 16, 17, 50, 100, 150, 240, 256]     # at K = 150 + 1 (two sources)
LINEAR_K = [1, 15, 16, 17, 101, 151, 301, 1024]                 # at n_out = 100
GRU_H = [1, 3, 4, 16, 61, 76, 77, 150, 153, 192]                # at kx = 150 + 1
GRU_KX = [1, 2, 3, 151]                                          # at H = 150


def linear_shapes():
    "(K, n_out) of every dense-layer case"
    return sorted(set([(151, n) for n in LINEAR_N_OUT] + [(k, 100) for k in LINEAR_K]))


def gru_shapes():
    "(kx, H) of every GRU-cell case"
    return sorted(set([(151, h) for h in GRU_H] + [(kx, 150) for kx in GRU_KX]))
