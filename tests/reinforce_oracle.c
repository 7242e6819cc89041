/*
 * TEST INFRASTRUCTURE ONLY -- CPU restatement of model type `reinforce` as the library's persistent kernel runs it
 * (include/pdp_b200.h pdp_set_reinforce) on top of the C oracle.  The oracle (oracle/pdp_oracle.c) is included as it is;
 * this file restates the loop of oracle/pdp_oracle.py reinforce_run (reference solver.py:355-386 with ReinforceDecimator,
 * ReinforcePredictor and _update_solution) with the oracle's own smooth-max and sparse_max (per-problem min, strict = 0),
 * the trainer's termination with `-b` replicas, and per-problem freeze iterations.
 */
#include "../oracle/pdp_oracle.c"

/* Runs up to T iterations from the oracle's current state (the caller has simplified and set the state: q3/fs2 are the
 * decimator state, pq3/pfs2 the propagator state).  coins [T]; check_termination: the active-mask semantics (retire test,
 * blend, predictor, CNF check); merged_out: NULL or [T][V], the merged prediction of every executed iteration (with
 * check_termination); freeze_out: NULL or int32 [B], the 1-based iteration at which each problem retired, -1 if never.
 * On return q3/fs2 (= pq3/pfs2) hold the final state and o->sol the last merged prediction.  Returns the iterations run. */
int64_t rf_run(ora_t* o, int64_t T, float pi, float p_dec, const float* coins, int check_termination, int batch_replication,
               float* merged_out, int32_t* freeze_out) {
    const int64_t E = o->E, V = o->V, B = o->B;
    const int rep = batch_replication > 1 ? batch_replication : 1;
    compute_edge_mask(o);
    double em_sum = 0, nav = 0;
    for (int64_t e = 0; e < E; ++e) em_sum += o->em[e];
    for (int64_t i = 0; i < V; ++i) nav += o->av[i];
    const int em_partial = em_sum < (double)E;
    for (int64_t b = 0; b < B; ++b) { o->active[b] = 1; if (freeze_out) freeze_out[b] = -1; }
    float* nq = ALLOC(float, 3 * E); float* nf = ALLOC(float, 2 * E);
    float* ps = ALLOC(float, V); float* ns = ALLOC(float, V);
    float* d = ALLOC(float, E); float* sd = ALLOC(float, V); float* db = ALLOC(float, B);
    float* score = ALLOC(float, V); float* solved = ALLOC(float, B); float* nun = ALLOC(float, B);
    int has_prev = 0;
    int64_t t = 0;
    while (t < T) {
        /* 1. SurveyPropagator with pi; the edge mask rides in the decimator state from the second iteration on */
        sp_step_core(o, o->q3, o->fs2, (t > 0 && em_partial) ? o->em : NULL, o->pq3, o->pfs2,
                     check_termination ? o->active : NULL, pi, nq, nf, o->tE1, o->tE2, o->tF1, ps, ns);
        const int64_t it = ++t;
        /* 2. ReinforceDecimator retire test (pdp_decimate.py:207-215) */
        if (check_termination && has_prev && nav > 0) {
            for (int64_t e = 0; e < E; ++e) {
                d[e] = fabsf(o->prev[e] - nf[2 * e]);
                if (it > 1) d[e] = d[e] * o->em[e];     /* sat_problem._edge_mask is set after the first iteration */
            }
            smooth_max_var(o, d, sd);
            for (int64_t i = 0; i < V; ++i) sd[i] = sd[i] * o->av[i];
            sparse_max_batch(o, sd, db);
            for (int64_t b = 0; b < B; ++b)
                if (o->active[b] && db[b] <= 0.01f) { o->active[b] = 0; if (freeze_out) freeze_out[b] = (int32_t)it; }
        }
        for (int64_t e = 0; e < E; ++e) o->prev[e] = nf[2 * e];
        has_prev = 1;
        /* 3. the coin: external forces from the SP biases (pdp_decimate.py:218-233) */
        if (coins[it - 1] < p_dec) {
            ora_score(o, nf, o->af, pi, score);
            for (int64_t e = 0; e < E; ++e) {
                const float sg = sgnf(score[o->evar[e]]);
                if (!check_termination) { nf[2 * e + 1] = sg; continue; }
                const float m = (float)o->active[o->bvm[o->evar[e]]];
                nf[2 * e + 1] = m * sg + (1.f - m) * nf[2 * e + 1];
            }
        }
        memcpy(o->q3, nq, sizeof(float) * 3 * (size_t)E); memcpy(o->fs2, nf, sizeof(float) * 2 * (size_t)E);
        memcpy(o->pq3, nq, sizeof(float) * 3 * (size_t)E); memcpy(o->pfs2, nf, sizeof(float) * 2 * (size_t)E);
        if (!check_termination) continue;
        /* 4. ReinforcePredictor + _update_solution (pdp_predict.py:221-226, solver.py:388-399) */
        for (int64_t i = 0; i < V; ++i) {
            float f = 0.f;
            for (int64_t p = o->vptr[i]; p < o->vptr[i + 1]; ++p) f += nf[2 * o->vedge[p] + 1];
            const float merged = o->av[i] * ((f > 0.f) ? 1.f : 0.f) + (1.f - o->av[i]) * o->sol[i];
            if (o->av[i] == 1.f) o->sol[i] = merged;
            if (merged_out) merged_out[(it - 1) * V + i] = merged;
        }
        /* 5. trainer.py:150-162: a solved replica retires every replica of its problem */
        ora_cnf_eval(o, o->sol, solved, nun);
        const int64_t B0 = B / rep;
        int64_t na = 0;
        for (int64_t j = 0; j < B0; ++j) {
            int any = 0;
            for (int r = 0; r < rep; ++r) any |= solved[r * B0 + j] > 0.5f;
            for (int r = 0; r < rep; ++r) {
                const int64_t b = r * B0 + j;
                if (any && o->active[b]) { o->active[b] = 0; if (freeze_out) freeze_out[b] = (int32_t)it; }
                na += o->active[b];
            }
        }
        if (na == 0) break;
    }
    o->iters_done += t;
    free(nq); free(nf); free(ps); free(ns); free(d); free(sd); free(db); free(score); free(solved); free(nun);
    return t;
}
