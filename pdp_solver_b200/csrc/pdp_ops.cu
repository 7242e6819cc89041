// pdp_ops.cu -- stateless operators in the caller's edge order (the reference's operator interface) and
// the import/export of the solver state held by a context.
#include <cub/cub.cuh>

#include "pdp_device.cuh"

namespace {

// ------------------------------------------------------------------------------------------------
// SatCNFEvaluator.forward (util.py:210-236)
// ------------------------------------------------------------------------------------------------
__global__ void k_cnf_eval_count(pdp_graph g, pdp_state s, const float* __restrict__ pred) {
    // s.conflicts counts clauses, s.energy counts satisfied clauses (both zero on entry, reset on exit)
    int last_b = -1, n_all = 0, n_sat = 0;
    WARP_STRIDED(a, g.F) {
        if (a >= g.F) continue;
        const int b = g.bfm[a];
        if (b != last_b) {
            if (last_b >= 0) { atomicAdd(&s.conflicts[last_b], n_all); atomicAdd(&s.energy[last_b], n_sat); }
            last_b = b; n_all = 0; n_sat = 0;
        }
        n_all += 1; n_sat += clause_satisfied(g.c_var, g.cl_ptr[a], g.cl_ptr[a + 1], pred) ? 1 : 0;
    }
    if (last_b >= 0) { atomicAdd(&s.conflicts[last_b], n_all); atomicAdd(&s.energy[last_b], n_sat); }
}

__global__ void k_cnf_eval_finish(pdp_graph g, pdp_state s, float* solved, float* n_unsat) {
    for (int64_t b = gtid(); b < g.B; b += gthreads()) {
        const int all = s.conflicts[b], sat = s.energy[b];
        solved[b] = (all == sat) ? 1.f : 0.f;
        n_unsat[b] = (float)(all - sat);
        s.conflicts[b] = 0; s.energy[b] = 0;
    }
}

// ------------------------------------------------------------------------------------------------
// _compute_energy / _compute_energy_diff (solver.py:469-496), float masks like the reference's
// ------------------------------------------------------------------------------------------------
__global__ void k_energy(pdp_graph g, const float* __restrict__ asg, const float* __restrict__ av,
                         const float* __restrict__ af, float* energy, float* unsat_fn, float* agg_out, float* deg_out) {
    WARP_STRIDED(a, g.F) {
        if (a >= g.F) continue;
        float agg = 0.f, deg = 0.f;
        for (int c = g.cl_ptr[a]; c < g.cl_ptr[a + 1]; ++c) {
            const uint32_t w = g.c_var[c];
            const int v = (int)(w & PDP_IDX_MASK);
            const float sg = (w & PDP_SIGN_BIT) ? -1.f : 1.f;
            agg += sg * (asg[v] * av[v]);
            deg += av[v];
        }
        if (agg_out) { agg_out[a] = agg; deg_out[a] = deg; }
        if (unsat_fn) {
            const float u = ((agg == -deg) ? 1.f : 0.f) * af[a];
            unsat_fn[a] = u;
            if (u != 0.f) atomicAdd(&energy[g.bfm[a]], u);   // small integers: exact in any order
        }
    }
}

__global__ void k_energy_diff(pdp_graph g, const float* __restrict__ asg, const float* __restrict__ av,
                              const float* __restrict__ em, const float* __restrict__ agg, const float* __restrict__ deg,
                              float* delta) {
    WARP_STRIDED(i, g.V) {
        if (i >= g.V) continue;
        float d = 0.f;
        const float lit0 = asg[i] * av[i];
        for (int p = g.var_ptr[i]; p < g.var_ptr[i + 1]; ++p) {
            const int a = g.v_cls[p];
            const float dist = ((g.v_cedge[p] & PDP_SIGN_BIT) ? -1.f : 1.f) * lit0;
            const float others = agg[a] - dist;
            const float crit = ((others == (1.f - deg[a])) ? 1.f : 0.f) * em[g.v_orig[p]];
            d += crit * dist;
        }
        delta[i] = d;
    }
}

// ------------------------------------------------------------------------------------------------
// SurveyPropagator.forward in the caller's edge order (pdp_propagate.py:139-221)
// ------------------------------------------------------------------------------------------------
// xlog / ext_in (nullable): the adaptor outputs of the neural variant (pdp_propagate.py:163-164,179-182) --
// the variable->clause message already in the log domain, the external force column
__global__ void k_sp_step_clause(pdp_graph g, const float* __restrict__ dq3, const float* __restrict__ em,
                                 const float* __restrict__ pfs2, const float* __restrict__ dfs2,
                                 const uint8_t* __restrict__ active, float* out_fs2,
                                 const float* __restrict__ xlog, const float* __restrict__ ext_in) {
    WARP_STRIDED(a, g.F) {
        if (a >= g.F) continue;
        const int beg = g.cl_ptr[a], end = g.cl_ptr[a + 1];
        float tot = 0.f;
        for (int c = beg; c < end; ++c) {
            const int e = g.c_orig[c];
            float v = xlog ? xlog[e] : L40(dq3[3 * (int64_t)e]);
            if (em) v = v * em[e];
            tot += v;
        }
        for (int c = beg; c < end; ++c) {
            const int e = g.c_orig[c];
            float v = xlog ? xlog[e] : L40(dq3[3 * (int64_t)e]);
            if (em) v = v * em[e];
            const float mask = active ? (float)active[g.bvm[g.c_var[c] & PDP_IDX_MASK]] : 1.f;
            out_fs2[2 * (int64_t)e] = mask * X30(tot - v) + (1.f - mask) * pfs2[2 * (int64_t)e];
            out_fs2[2 * (int64_t)e + 1] = ext_in ? ext_in[e] : dfs2[2 * (int64_t)e + 1];
        }
    }
}

__global__ void k_sp_step_var(pdp_graph g, const float* __restrict__ dfs2, const float* __restrict__ em,
                              const float* __restrict__ pq3, const uint8_t* __restrict__ active, float pi, float* out_q3,
                              const float* __restrict__ eta_in, const float* __restrict__ ext_in) {
    WARP_STRIDED(i, g.V) {
        if (i >= g.V) continue;
        const int beg = g.var_ptr[i], end = g.var_ptr[i + 1];
        const float mask = active ? (float)active[g.bvm[i]] : 1.f;
        float P = 0.f, N = 0.f;
        for (int p = beg; p < end; ++p) {
            const int e = g.v_orig[p];
            float y = L40_1m(eta_in ? eta_in[e] : dfs2[2 * (int64_t)e]);
            if (em) y = y * em[e];
            const bool neg = (g.v_cedge[p] & PDP_SIGN_BIT) != 0u;
            P += (neg ? 0.f : 1.f) * y;
            N += (neg ? 1.f : 0.f) * y;
        }
        for (int p = beg; p < end; ++p) {
            const int64_t e = g.v_orig[p];
            float y = L40_1m(eta_in ? eta_in[e] : dfs2[2 * e]);
            if (em) y = y * em[e];
            float u, v, d;
            sp_var_update(P, N, y, (g.v_cedge[p] & PDP_SIGN_BIT) ? -1.f : 1.f, ext_in ? ext_in[e] : dfs2[2 * e + 1], pi, u, v, d);
            out_q3[3 * e + 0] = mask * u + (1.f - mask) * pq3[3 * e + 0];
            out_q3[3 * e + 1] = mask * v + (1.f - mask) * pq3[3 * e + 1];
            out_q3[3 * e + 2] = mask * d + (1.f - mask) * pq3[3 * e + 2];
        }
    }
}

// node sums of [E,C] edge rows (ascending edge order, fp32) and the leave-one-out gather back to the edges.
// A warp walks the channels of one node (coalesced rows).
__global__ void k_edge_aggregate(pdp_graph g, int by_variable, const float* __restrict__ state, int C, float* node_sum, float* edge_loo) {
    const int64_t nodes = by_variable ? g.V : g.F;
    const int32_t* ptr = by_variable ? g.var_ptr : g.cl_ptr;
    const int32_t* orig = by_variable ? g.v_orig : g.c_orig;
    for (int64_t node = gwarp(); node < nodes; node += gwarps()) {
        const int beg = ptr[node], end = ptr[node + 1];
        for (int ch = lane_id(); ch < C; ch += 32) {
            float acc = 0.f;
            for (int k = beg; k < end; ++k) acc += state[(int64_t)orig[k] * C + ch];
            node_sum[node * C + ch] = acc;
            if (edge_loo) for (int k = beg; k < end; ++k) { const int64_t e = orig[k]; edge_loo[e * C + ch] = acc - state[e * C + ch]; }
        }
    }
}

// SurveyScorer.forward (pdp_predict.py:155-192), float clause mask
__global__ void k_score(pdp_graph g, const float* __restrict__ fs2, const float* __restrict__ af, float pi, float* score) {
    WARP_STRIDED(i, g.V) {
        if (i >= g.V) continue;
        float extsum = 0.f, ps = 0.f, ns = 0.f, as = 0.f;
        for (int p = g.var_ptr[i]; p < g.var_ptr[i + 1]; ++p) {
            const int64_t e = g.v_orig[p];
            extsum += fs2[2 * e + 1];
            const float f = L10(1.f - fs2[2 * e]) * af[g.v_cls[p]];
            const bool neg = (g.v_cedge[p] & PDP_SIGN_BIT) != 0u;
            ps += (neg ? 0.f : 1.f) * f;
            ns += (neg ? 1.f : 0.f) * f;
            as += f;
        }
        score[i] = sp_score_tail(ps, ns, as, sgnf(extsum), pi);
    }
}

// ------------------------------------------------------------------------------------------------
// state import / export
// ------------------------------------------------------------------------------------------------
__global__ void k_load_state(pdp_graph g, pdp_state s, const float* __restrict__ dq3, const float* __restrict__ dfs2, int buf) {
    for (int64_t p = gtid(); p < g.E; p += gthreads()) {
        const int64_t e = g.v_orig[p];
        const int qp = g.p_qpos[p];
        s.qu[qp] = dq3[3 * e]; s.qs[qp] = dq3[3 * e + 1]; s.qd[qp] = dq3[3 * e + 2];
        const float eta = dfs2[2 * e];
        const float ext = dfs2[2 * e + 1];
        s.eta[buf][g.p_vpos[p]] = eta; s.ext[p] = ext;
        // reinforce runs the blocked passes only on forces that are uniform over each variable's edges (NaN counts as equal)
        const float e0 = dfs2[2 * (int64_t)g.v_orig[g.var_ptr[g.c_var[g.v_cedge[p] & PDP_IDX_MASK] & PDP_IDX_MASK]] + 1];
        if (!(ext == e0 || (ext != ext && e0 != e0))) s.ctrl[CTRL_RF_MIXED] = 1;
        // the blocked passes borrow the sign bits of the messages they read and write: messages that arrive with one (not
        // a probability) go through the generic passes until no message can carry a sign any more -- the first iteration
        // reads them, the second reads the q the first derived from them (a survey below 0 makes exp(opp) > 1 and q < 0);
        // a clause-side survey is an exponential and a q derived from surveys >= 0 is >= +0
        if ((__float_as_uint(eta) | __float_as_uint(dq3[3 * e])) >> 31) s.ctrl[CTRL_GEN_ITERS] = 2;
    }
}

// the predict path's initial messages are constants (reference pdp_predict.py:203-206): no gather
__global__ void k_load_state_const(pdp_graph g, pdp_state s, float qu, float qs, float qd, float eta, float ext, int buf) {
    for (int64_t p = gtid(); p < g.E; p += gthreads()) {
        s.qu[p] = qu; s.qs[p] = qs; s.qd[p] = qd; s.eta[buf][p] = eta; s.ext[p] = ext;
    }
    if (gtid() == 0 && ((__float_as_uint(eta) | __float_as_uint(qu)) >> 31)) s.ctrl[CTRL_GEN_ITERS] = 2;
}

// thread per variable; when the [E,3] state was not tracked every iteration, q_s and q_* are
// re-derived from the previous surveys with the current masks (materialised once, on exit)
__global__ void k_store_state(pdp_graph g, pdp_state s, float* out_q3, float* out_fs2, int iter, int tracked, float pi) {
    WARP_STRIDED(i, g.V) {
        if (i >= g.V) continue;
        const int b = g.bvm[i];
        const int fz = s.freeze_iter[b];
        const int last = (fz >= 0) ? fz : iter;
        const int buf = last & 1;
        const int beg = g.var_ptr[i], end = g.var_ptr[i + 1];
        const bool rebuild = (!tracked) && last >= 1;
        const bool stashed = last == s.rf_coin_iter[b];   // reinforce: the coin after the sweep of `last` changed the forces
        float P = 0.f, N = 0.f;
        const bool um = (last >= 2) && s.masked[b];
        const float avi = (float)s.av[i];
        if (rebuild) {
            for (int p = beg; p < end; ++p) {
                float y = L40_1m(s.eta[buf ^ 1][g.p_vpos[p]]);
                if (um) y = y * (avi * (float)s.af[g.v_cls[p]]);
                const bool neg = (g.v_cedge[p] & PDP_SIGN_BIT) != 0u;
                P += (neg ? 0.f : 1.f) * y;
                N += (neg ? 1.f : 0.f) * y;
            }
        }
        for (int p = beg; p < end; ++p) {
            const int64_t e = g.v_orig[p];
            const int qp = g.p_qpos[p], vp = g.p_vpos[p];
            float u = s.qu[qp], v = s.qs[qp], d = s.qd[qp];
            if (rebuild) {
                float y = L40_1m(s.eta[buf ^ 1][vp]);
                if (um) y = y * (avi * (float)s.af[g.v_cls[p]]);
                float uu;
                sp_var_update(P, N, y, (g.v_cedge[p] & PDP_SIGN_BIT) ? -1.f : 1.f, stashed ? s.qs[p] : s.ext[p], pi, uu, v, d);
            }
            if (out_q3) { out_q3[3 * e] = u; out_q3[3 * e + 1] = v; out_q3[3 * e + 2] = d; }
            if (out_fs2) { out_fs2[2 * e] = s.eta[buf][vp]; out_fs2[2 * e + 1] = s.ext[p]; }
        }
    }
}

__global__ void k_set_masks(pdp_graph g, pdp_state s, const float* av, const float* af, const float* sol) {
    const int64_t n = max(max(g.V, g.F), g.B);
    for (int64_t i = gtid(); i < n; i += gthreads()) {
        if (i < g.V) { if (av) s.av[i] = (av[i] != 0.f) ? 1 : 0; if (sol) s.sol[i] = sol[i]; }
        if (i < g.F && af) s.af[i] = (af[i] != 0.f) ? 1 : 0;
        if (i < g.B) { s.masked[i] = 1; s.dirty[i] = 1; }
        if (i == 0) {
            s.ctrl[CTRL_ANY_DIRTY] = 1; s.ctrl[CTRL_CLOSED] = 0; s.ctrl[CTRL_NATIVE] = 0;   // masks from outside: closure unknown
            // node masks installed by the caller are part of the decimator state: the next sweep multiplies by the edge
            // mask they imply, as the reference does from the iteration after a mask changed (solver.py:370-374)
            if (av || af) { s.ctrl[CTRL_USE_MASK] = 1; s.ctrl[CTRL_EM_SET] = 1; }
        }
    }
}

// edge-mask bits from the node masks (after an external pdp_set_masks)
__global__ void k_clear_mask_bits(pdp_graph g) {
    for (int64_t wi = gtid(); wi < g.E / 32 + 1; wi += gthreads()) { g.vmask[wi] = 0u; g.qmask[wi] = 0u; }
}
__global__ void k_rebuild_mask_bits(pdp_graph g, pdp_state s) {
    for (int64_t c = gtid(); c < g.E; c += gthreads()) {
        const int p = g.c_pos[c];
        if (!(s.av[g.c_var[c] & PDP_IDX_MASK] && s.af[g.v_cls[p]])) mask_edge(g, cvpos(g, c), cqpos(g, c));
    }
}

__global__ void k_get_masks(pdp_graph g, pdp_state s, float* av, float* af, float* sol, float* is_sat, uint8_t* active, float* em) {
    const int64_t n = max(max(g.V, g.F), g.B);
    for (int64_t i = gtid(); i < n; i += gthreads()) {
        if (i < g.V) {
            if (av) av[i] = (float)s.av[i];
            if (sol) sol[i] = s.sol[i];
            if (em) for (int p = g.var_ptr[i]; p < g.var_ptr[i + 1]; ++p) em[g.v_orig[p]] = (float)s.av[i] * (float)s.af[g.v_cls[p]];
        }
        if (i < g.F && af) af[i] = (float)s.af[i];
        if (i < g.B) { if (is_sat) is_sat[i] = s.is_sat[i]; if (active) active[i] = s.active[i]; }
    }
}

__global__ void k_get_flags(pdp_graph g, pdp_state s, uint32_t* flags, int32_t* counters, int32_t* freeze) {
    for (int64_t b = gtid(); b < g.B; b += gthreads()) {
        if (flags) flags[b] = s.flags[b];
        if (counters) counters[b] = s.counters[b];
        if (freeze) freeze[b] = s.freeze_iter[b];
    }
}

struct U8ToInt {
    __host__ __device__ __forceinline__ int operator()(const uint8_t& x) const { return (int)x; }
};

__global__ void k_random_fill(pdp_graph g, pdp_state s, const float* __restrict__ draws) {
    for (int64_t i = gtid(); i < g.V; i += gthreads())
        if (s.av[i]) s.sol[i] = draws[s.scan_tmp[i]];
    if (gtid() == 0) s.ctrl[CTRL_NATIVE] = 0;   // active variables now carry values: an active clause may be satisfied
}

// _deduplicate (solver.py:401-431)
__global__ void k_dedup_energy(pdp_graph g, pdp_state s, const float* __restrict__ pred) {
    WARP_STRIDED(a, g.F) {
        if (a >= g.F) continue;
        if (!s.af[a]) continue;
        float agg = 0.f, deg = 0.f;
        for (int c = g.cl_ptr[a]; c < g.cl_ptr[a + 1]; ++c) {
            const uint32_t w = g.c_var[c];
            const int v = (int)(w & PDP_IDX_MASK);
            const float avv = (float)s.av[v];
            agg += ((w & PDP_SIGN_BIT) ? -1.f : 1.f) * ((2.f * pred[v] - 1.0f) * avv);
            deg += avv;
        }
        if (agg == -deg) atomicAdd(&s.energy[g.bfm[a]], 1);
    }
}

__global__ void k_dedup_pick(pdp_graph g, pdp_state s, int rep, int32_t* winner) {
    const int64_t B0 = g.B / rep;
    for (int64_t j = gtid(); j < B0; j += gthreads()) {
        int best = 0, be = s.energy[j];
        for (int r = 1; r < rep; ++r) { const int en = s.energy[(int64_t)r * B0 + j]; if (en < be) { be = en; best = r; } }
        winner[j] = best;
    }
}

__global__ void k_dedup_gather(pdp_graph g, pdp_state s, int rep, const float* __restrict__ pred, const int32_t* __restrict__ winner,
                               float* out) {
    const int64_t V0 = g.V / rep;
    for (int64_t i = gtid(); i < g.V; i += gthreads()) {
        if (i < V0) out[i] = pred[(int64_t)winner[g.bvm[i]] * V0 + i];
    }
    for (int64_t b = gtid(); b < g.B; b += gthreads()) s.energy[b] = 0;
}

}  // namespace

#define GRID(n) pdp_grid((n), 256, ctx->num_sms), 256, 0, stream
#define NEED(ctx, cond, msg) do { if (!(ctx)) { pdp_set_error("null context"); return PDP_ERR_ARG; } if (!(cond)) { pdp_set_error(msg); return PDP_ERR_ARG; } } while (0)

extern "C" int pdp_cnf_eval(pdp_ctx* ctx, const float* d_pred, float* d_solved, float* d_n_unsat, void* stream_) {
    NEED(ctx, (d_pred || ctx->g.V == 0) && d_solved && d_n_unsat, "pdp_cnf_eval: null argument");
    cudaStream_t stream = (cudaStream_t)stream_;
    if (ctx->g.F > 0) { k_cnf_eval_count<<<GRID(ctx->g.F)>>>(ctx->g, ctx->s, d_pred); PDP_LAUNCH_CHECK(ctx); }
    k_cnf_eval_finish<<<GRID(ctx->g.B)>>>(ctx->g, ctx->s, d_solved, d_n_unsat);
    PDP_LAUNCH_CHECK(ctx);
    return PDP_OK;
}

// ---- context-free CNF check on the caller's edge list (SatCNFEvaluator called on a batch nobody built a context for)
namespace {
__global__ void k_edges_mark_sat(const int32_t* __restrict__ evar, const int32_t* __restrict__ ecls, const float* __restrict__ sign,
                                 const float* __restrict__ pred, int64_t E, int64_t V, int64_t F, uint8_t* clause_sat, int32_t* bad) {
    for (int64_t e = gtid(); e < E; e += gthreads()) {
        const int32_t v = evar[e], a = ecls[e];
        if (v < 0 || v >= V || a < 0 || a >= F) { *bad = 1; continue; }
        if (literal_true(sign[e], pred[v])) clause_sat[a] = 1;      // util.py:221-228 (benign race: every writer stores 1)
    }
}
__global__ void k_edges_count_unsat(const uint8_t* __restrict__ clause_sat, const int32_t* __restrict__ bfm, int64_t F, int64_t B,
                                    int32_t* n_unsat, int32_t* bad) {
    for (int64_t a = gtid(); a < F; a += gthreads()) {
        const int32_t b = bfm[a];
        if (b < 0 || b >= B) { *bad = 1; continue; }
        if (!clause_sat[a]) atomicAdd(&n_unsat[b], 1);
    }
}
__global__ void k_edges_finish(const int32_t* __restrict__ n_unsat, int64_t B, float* solved, float* nun) {
    for (int64_t b = gtid(); b < B; b += gthreads()) { nun[b] = (float)n_unsat[b]; solved[b] = n_unsat[b] == 0 ? 1.f : 0.f; }
}
}  // namespace

extern "C" size_t pdp_cnf_eval_edges_scratch_bytes(int64_t F, int64_t B) {
    return (size_t)((F + 3) / 4 * 4) + sizeof(int32_t) * (size_t)(B + 1);
}

extern "C" int pdp_cnf_eval_edges(const int32_t* d_graph_map, const float* d_edge_feature, const int32_t* d_bfm,
                                  int64_t E, int64_t V, int64_t F, int64_t B, const float* d_pred,
                                  float* d_solved, float* d_n_unsat, void* d_scratch, void* stream_) {
    if (E < 0 || V < 0 || F < 0 || B < 0 || (B > 0 && (!d_solved || !d_n_unsat)) || !d_scratch || (E > 0 && (!d_graph_map || !d_edge_feature || !d_pred)) ||
        (F > 0 && !d_bfm)) { pdp_set_error("pdp_cnf_eval_edges: bad argument"); return PDP_ERR_ARG; }
    cudaStream_t stream = (cudaStream_t)stream_;
    int dev = 0, nsm = 148;
    PDP_CUDA_CHECK(cudaGetDevice(&dev));
    PDP_CUDA_CHECK(cudaDeviceGetAttribute(&nsm, cudaDevAttrMultiProcessorCount, dev));
    uint8_t* clause_sat = reinterpret_cast<uint8_t*>(d_scratch);
    int32_t* n_unsat = reinterpret_cast<int32_t*>(clause_sat + (F + 3) / 4 * 4);
    int32_t* bad = n_unsat + B;
    PDP_CUDA_CHECK(cudaMemsetAsync(d_scratch, 0, pdp_cnf_eval_edges_scratch_bytes(F, B), stream));
    if (E > 0) k_edges_mark_sat<<<pdp_grid(E, 256, nsm), 256, 0, stream>>>(d_graph_map, d_graph_map + E, d_edge_feature, d_pred, E, V, F, clause_sat, bad);
    if (F > 0) k_edges_count_unsat<<<pdp_grid(F, 256, nsm), 256, 0, stream>>>(clause_sat, d_bfm, F, B, n_unsat, bad);
    if (B > 0) k_edges_finish<<<pdp_grid(B, 256, nsm), 256, 0, stream>>>(n_unsat, B, d_solved, d_n_unsat);
    PDP_CUDA_CHECK(cudaGetLastError());
    return PDP_OK;
}

extern "C" int pdp_energy(pdp_ctx* ctx, const float* d_asg, const float* d_av, const float* d_af, float* d_energy,
                          float* d_unsat_fn, void* stream_) {
    NEED(ctx, (d_asg && d_av || ctx->g.V == 0) && (d_af && d_unsat_fn || ctx->g.F == 0) && d_energy, "pdp_energy: null argument");
    cudaStream_t stream = (cudaStream_t)stream_;
    PDP_CUDA_CHECK(cudaMemsetAsync(d_energy, 0, sizeof(float) * (size_t)ctx->g.B, stream));
    if (ctx->g.F > 0) { k_energy<<<GRID(ctx->g.F)>>>(ctx->g, d_asg, d_av, d_af, d_energy, d_unsat_fn, nullptr, nullptr); PDP_LAUNCH_CHECK(ctx); }
    return PDP_OK;
}

extern "C" int pdp_energy_diff(pdp_ctx* ctx, const float* d_asg, const float* d_av, const float* d_em, float* d_delta, void* stream_) {
    NEED(ctx, (d_asg && d_av && d_delta || ctx->g.V == 0) && (d_em || ctx->g.E == 0), "pdp_energy_diff: null argument");
    cudaStream_t stream = (cudaStream_t)stream_;
    float* agg = reinterpret_cast<float*>(ctx->s.ws_true);
    float* deg = reinterpret_cast<float*>(ctx->s.ws_deg);
    if (ctx->g.F > 0) { k_energy<<<GRID(ctx->g.F)>>>(ctx->g, d_asg, d_av, nullptr, nullptr, nullptr, agg, deg); PDP_LAUNCH_CHECK(ctx); }
    if (ctx->g.V > 0) { k_energy_diff<<<GRID(ctx->g.V)>>>(ctx->g, d_asg, d_av, d_em, agg, deg, d_delta); PDP_LAUNCH_CHECK(ctx); }
    return PDP_OK;
}

extern "C" int pdp_sp_step(pdp_ctx* ctx, const float* d_dec_q3, const float* d_dec_fs2, const float* d_edge_mask,
                           const float* d_prop_q3, const float* d_prop_fs2, const uint8_t* d_active, float pi,
                           float* d_out_q3, float* d_out_fs2, void* stream_) {
    NEED(ctx, (d_dec_q3 && d_dec_fs2 && d_out_q3 && d_out_fs2) || ctx->g.E == 0, "pdp_sp_step: null argument");
    cudaStream_t stream = (cudaStream_t)stream_;
    const float* pq = d_prop_q3 ? d_prop_q3 : d_dec_q3;
    const float* pf = d_prop_fs2 ? d_prop_fs2 : d_dec_fs2;
    if (ctx->g.F > 0) { k_sp_step_clause<<<GRID(ctx->g.F)>>>(ctx->g, d_dec_q3, d_edge_mask, pf, d_dec_fs2, d_active, d_out_fs2, nullptr, nullptr); PDP_LAUNCH_CHECK(ctx); }
    if (ctx->g.V > 0) { k_sp_step_var<<<GRID(ctx->g.V)>>>(ctx->g, d_dec_fs2, d_edge_mask, pq, d_active, pi, d_out_q3, nullptr, nullptr); PDP_LAUNCH_CHECK(ctx); }
    return PDP_OK;
}

extern "C" int pdp_sp_step_adapted(pdp_ctx* ctx, const float* d_x_log, const float* d_eta_in, const float* d_ext_in,
                                   const float* d_edge_mask, const float* d_prop_q3, const float* d_prop_fs2,
                                   const uint8_t* d_active, float pi, float* d_out_q3, float* d_out_fs2, void* stream_) {
    NEED(ctx, (d_x_log && d_eta_in && d_ext_in && d_prop_q3 && d_prop_fs2 && d_out_q3 && d_out_fs2) || ctx->g.E == 0, "pdp_sp_step_adapted: null argument");
    cudaStream_t stream = (cudaStream_t)stream_;
    if (ctx->g.F > 0) { k_sp_step_clause<<<GRID(ctx->g.F)>>>(ctx->g, nullptr, d_edge_mask, d_prop_fs2, nullptr, d_active, d_out_fs2, d_x_log, d_ext_in); PDP_LAUNCH_CHECK(ctx); }
    if (ctx->g.V > 0) { k_sp_step_var<<<GRID(ctx->g.V)>>>(ctx->g, nullptr, d_edge_mask, d_prop_q3, d_active, pi, d_out_q3, d_eta_in, d_ext_in); PDP_LAUNCH_CHECK(ctx); }
    return PDP_OK;
}

// torch.mm(mask[N,E], state[E,C]) of MessageAggregator (util.py:60): per node the sum of its edges' rows in
// ascending edge order; optionally the gather back to the edges minus the own row (leave one out, util.py:62-68)
extern "C" int pdp_edge_aggregate(pdp_ctx* ctx, int32_t by_variable, const float* d_state, int32_t channels, float* d_node_sum,
                                  float* d_edge_loo, void* stream_) {
    NEED(ctx, d_state && d_node_sum && channels > 0, "pdp_edge_aggregate: bad argument");
    cudaStream_t stream = (cudaStream_t)stream_;
    const int64_t nodes = by_variable ? ctx->g.V : ctx->g.F;
    if (nodes > 0) {
        k_edge_aggregate<<<GRID(nodes * (int64_t)std::min(channels, 32))>>>(ctx->g, by_variable, d_state, channels, d_node_sum, d_edge_loo);
        PDP_LAUNCH_CHECK(ctx);
    }
    return PDP_OK;
}

extern "C" int pdp_score(pdp_ctx* ctx, const float* d_fs2, const float* d_af, float pi, float* d_score, void* stream_) {
    NEED(ctx, (d_fs2 || ctx->g.E == 0) && (d_af || ctx->g.F == 0) && (d_score || ctx->g.V == 0), "pdp_score: null argument");
    cudaStream_t stream = (cudaStream_t)stream_;
    if (ctx->g.V > 0) { k_score<<<GRID(ctx->g.V)>>>(ctx->g, d_fs2, d_af, pi, d_score); PDP_LAUNCH_CHECK(ctx); }
    return PDP_OK;
}

extern "C" int pdp_load_state(pdp_ctx* ctx, const float* d_prop_q3, const float* d_prop_fs2, const float* d_dec_q3,
                              const float* d_dec_fs2, void* stream_) {
    (void)d_prop_q3; (void)d_prop_fs2;   // only reachable through the frozen-problem blend; every problem starts active
    NEED(ctx, (d_dec_q3 && d_dec_fs2) || ctx->g.E == 0, "pdp_load_state: null argument");
    cudaStream_t stream = (cudaStream_t)stream_;
    PDP_CUDA_CHECK(cudaMemsetAsync(ctx->s.ctrl + CTRL_GEN_ITERS, 0, sizeof(int32_t), stream));
    PDP_CUDA_CHECK(cudaMemsetAsync(ctx->s.ctrl + CTRL_RF_MIXED, 0, sizeof(int32_t), stream));
    if (ctx->g.E > 0) { k_load_state<<<GRID(ctx->g.E)>>>(ctx->g, ctx->s, d_dec_q3, d_dec_fs2, 0); PDP_LAUNCH_CHECK(ctx); }
    return PDP_OK;
}

extern "C" int pdp_load_state_const(pdp_ctx* ctx, float qu, float qs, float qd, float eta, float ext, void* stream_) {
    NEED(ctx, true, "");
    cudaStream_t stream = (cudaStream_t)stream_;
    PDP_CUDA_CHECK(cudaMemsetAsync(ctx->s.ctrl + CTRL_GEN_ITERS, 0, sizeof(int32_t), stream));
    PDP_CUDA_CHECK(cudaMemsetAsync(ctx->s.ctrl + CTRL_RF_MIXED, 0, sizeof(int32_t), stream));
    if (ctx->g.E > 0) { k_load_state_const<<<GRID(ctx->g.E)>>>(ctx->g, ctx->s, qu, qs, qd, eta, ext, 0); PDP_LAUNCH_CHECK(ctx); }
    return PDP_OK;
}

extern "C" int pdp_store_state(pdp_ctx* ctx, float* d_out_q3, float* d_out_fs2, void* stream_) {
    NEED(ctx, d_out_q3 || d_out_fs2 || ctx->g.E == 0, "pdp_store_state: null argument");
    cudaStream_t stream = (cudaStream_t)stream_;
    int32_t h[2] = {0, 0};
    PDP_CUDA_CHECK(cudaMemcpyAsync(h, ctx->s.ctrl + CTRL_ITER, sizeof(int32_t), cudaMemcpyDeviceToHost, stream));
    PDP_CUDA_CHECK(cudaStreamSynchronize(stream));
    if (ctx->g.V > 0) {
        k_store_state<<<GRID(ctx->g.V)>>>(ctx->g, ctx->s, d_out_q3, d_out_fs2, h[0], ctx->full_state_tracked, ctx->last_pi);
        PDP_LAUNCH_CHECK(ctx);
    }
    return PDP_OK;
}

extern "C" int pdp_set_masks(pdp_ctx* ctx, const float* d_av, const float* d_af, const float* d_sol, void* stream_) {
    NEED(ctx, true, "");
    cudaStream_t stream = (cudaStream_t)stream_;
    const int64_t n = std::max(std::max(ctx->g.V, ctx->g.F), std::max(ctx->g.B, (int64_t)1));
    k_set_masks<<<GRID(n)>>>(ctx->g, ctx->s, d_av, d_af, d_sol);
    PDP_LAUNCH_CHECK(ctx);
    if (ctx->g.E > 0 && (d_av || d_af)) {
        k_clear_mask_bits<<<GRID(ctx->g.E / 32 + 1)>>>(ctx->g);
        PDP_LAUNCH_CHECK(ctx);
        k_rebuild_mask_bits<<<GRID(ctx->g.E)>>>(ctx->g, ctx->s);
        PDP_LAUNCH_CHECK(ctx);
    }
    return PDP_OK;
}

// active_mask of _forward_core as a caller's termination callback left it (reference solver.py:376-384)
namespace {
__global__ void k_set_active(pdp_graph g, pdp_state s, const uint8_t* __restrict__ active) {
    int n = 0;
    for (int64_t b = gtid(); b < g.B; b += gthreads()) {
        const uint8_t a = active[b] ? 1 : 0;
        if (s.active[b] && !a) s.freeze_iter[b] = s.ctrl[CTRL_ITER];
        if (!s.active[b] && a) s.freeze_iter[b] = -1;
        n += (int)a - (int)s.active[b];
        s.active[b] = a;
    }
    if (n) atomicAdd(&s.ctrl[CTRL_NUM_ACTIVE], n);
}
}  // namespace
extern "C" int pdp_set_active(pdp_ctx* ctx, const uint8_t* d_active, void* stream_) {
    NEED(ctx, d_active || ctx->g.B == 0, "pdp_set_active: null argument");
    cudaStream_t stream = (cudaStream_t)stream_;
    if (ctx->g.B > 0) { k_set_active<<<GRID(ctx->g.B)>>>(ctx->g, ctx->s, d_active); PDP_LAUNCH_CHECK(ctx); }
    return PDP_OK;
}

extern "C" int pdp_get_masks(pdp_ctx* ctx, float* d_av, float* d_af, float* d_sol, float* d_is_sat, uint8_t* d_active,
                             float* d_em, void* stream_) {
    NEED(ctx, true, "");
    cudaStream_t stream = (cudaStream_t)stream_;
    const int64_t n = std::max(std::max(ctx->g.V, ctx->g.F), std::max(ctx->g.B, (int64_t)1));
    k_get_masks<<<GRID(n)>>>(ctx->g, ctx->s, d_av, d_af, d_sol, d_is_sat, d_active, d_em);
    PDP_LAUNCH_CHECK(ctx);
    return PDP_OK;
}

extern "C" int pdp_get_problem_flags(pdp_ctx* ctx, uint32_t* d_flags, int32_t* d_counters, int32_t* d_freeze, void* stream_) {
    NEED(ctx, true, "");
    cudaStream_t stream = (cudaStream_t)stream_;
    k_get_flags<<<GRID(ctx->g.B)>>>(ctx->g, ctx->s, d_flags, d_counters, d_freeze);
    PDP_LAUNCH_CHECK(ctx);
    return PDP_OK;
}

extern "C" int pdp_count_active_variables(pdp_ctx* ctx, int64_t* host_out, void* stream_) {
    NEED(ctx, host_out, "pdp_count_active_variables: null argument");
    cudaStream_t stream = (cudaStream_t)stream_;
    *host_out = 0;
    if (ctx->g.V == 0) return PDP_OK;
    cub::TransformInputIterator<int, U8ToInt, const uint8_t*> it(ctx->s.av, U8ToInt());
    size_t tb = ctx->cub_tmp_bytes;
    int* d_sum = ctx->s.scan_tmp + ctx->g.V;
    PDP_CUDA_CHECK(cub::DeviceReduce::Sum(ctx->cub_tmp, tb, it, d_sum, (int)ctx->g.V, stream));
    ctx->launches++;
    int h = 0;
    PDP_CUDA_CHECK(cudaMemcpyAsync(&h, d_sum, sizeof(int), cudaMemcpyDeviceToHost, stream));
    PDP_CUDA_CHECK(cudaStreamSynchronize(stream));
    *host_out = h;
    return PDP_OK;
}

extern "C" int pdp_random_fill(pdp_ctx* ctx, const float* d_draws, void* stream_) {
    NEED(ctx, d_draws || ctx->g.V == 0, "pdp_random_fill: null argument");
    cudaStream_t stream = (cudaStream_t)stream_;
    if (ctx->g.V == 0) return PDP_OK;
    cub::TransformInputIterator<int, U8ToInt, const uint8_t*> it(ctx->s.av, U8ToInt());
    size_t tb = ctx->cub_tmp_bytes;
    PDP_CUDA_CHECK(cub::DeviceScan::ExclusiveSum(ctx->cub_tmp, tb, it, ctx->s.scan_tmp, (int)ctx->g.V, stream));
    ctx->launches++;
    k_random_fill<<<GRID(ctx->g.V)>>>(ctx->g, ctx->s, d_draws);
    PDP_LAUNCH_CHECK(ctx);
    return PDP_OK;
}

extern "C" int pdp_deduplicate(pdp_ctx* ctx, int32_t rep, const float* d_pred, float* d_out, int32_t* d_winner, void* stream_) {
    NEED(ctx, (d_pred && d_out || ctx->g.V == 0) && d_winner && rep >= 1, "pdp_deduplicate: bad argument");
    if (ctx->g.B % rep || ctx->g.V % rep) { pdp_set_error("pdp_deduplicate: sizes not divisible by the replication factor"); return PDP_ERR_ARG; }
    cudaStream_t stream = (cudaStream_t)stream_;
    if (ctx->g.F > 0) { k_dedup_energy<<<GRID(ctx->g.F)>>>(ctx->g, ctx->s, d_pred); PDP_LAUNCH_CHECK(ctx); }
    k_dedup_pick<<<GRID(ctx->g.B)>>>(ctx->g, ctx->s, rep, d_winner);
    PDP_LAUNCH_CHECK(ctx);
    k_dedup_gather<<<GRID(std::max(ctx->g.V, ctx->g.B))>>>(ctx->g, ctx->s, rep, d_pred, d_winner, d_out);
    PDP_LAUNCH_CHECK(ctx);
    return PDP_OK;
}
