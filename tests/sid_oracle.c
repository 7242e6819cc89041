/*
 * TEST INFRASTRUCTURE ONLY -- CPU restatement of SP-inspired decimation (a fraction of each problem's active variables
 * fixed per decimation step; include/pdp_b200.h pdp_set_decimation_fraction / pdp_decimation_select) on top of the C
 * oracle.  The oracle (oracle/pdp_oracle.c) is included as it is; what differs is SequentialDecimator.forward, restated
 * below as sid_decimate with the fraction rule in place of the arg-max fix (K_b == 1 is that arg-max fix, unchanged), and
 * the loop that calls it (sid_iterate / sid_run).  Defined for strict = 0: the reference has no such mode to couple to.
 */
#include "../oracle/pdp_oracle.c"

/* ------------------------------------------------------------------------------------------ */
/* the rule: K_b = max(1, floor((double)f * A_b)); K_b == 1 the arg-max of pdp_decimate.py:152-171, else the first   */
/* min(K_b, #candidates) active variables with c > 0 by (c descending, index ascending)                               */
/* ------------------------------------------------------------------------------------------ */
static int valid_fraction(float f) { return f == f && f >= 0.f && f < 1.f; }

static int64_t sel_k(float f, float nav) {
    double k = floor((double)f * (double)nav);
    return k < 1.0 ? 1 : (int64_t)k;
}

typedef struct { float c; int64_t i; } cand_t;
static int cand_cmp(const void* a, const void* b) {
    const cand_t* x = (const cand_t*)a; const cand_t* y = (const cand_t*)b;
    if (x->c != y->c) return x->c > y->c ? -1 : 1;
    return x->i < y->i ? -1 : (x->i > y->i ? 1 : 0);
}

/* the decimation rule on coefficients c [V] (>= 0, |score| * active * converged) and scores [V]:
 * sel[b] != 0 marks the problems the caller selected (converged, active); nav[b] = active variables of b.
 * Writes sign(score) of the taken variables into asg (which the caller zeroed) and, when `trace`, records them. */
static void decimation_rule(ora_t* o, const float* c, const float* score, const int* sel, const float* nav, float frac,
                            float* asg, int trace) {
    const int64_t V = o->V, B = o->B;
    int64_t* mi = (int64_t*)malloc(sizeof(int64_t) * (size_t)(B > 0 ? B : 1));
    int64_t* K = (int64_t*)malloc(sizeof(int64_t) * (size_t)(B > 0 ? B : 1));
    int64_t* ptr = (int64_t*)calloc((size_t)(B + 1), sizeof(int64_t));
    sparse_argmax_batch(o, c, mi);
    for (int64_t b = 0; b < B; ++b) K[b] = sel[b] ? sel_k(frac, nav[b]) : 0;
    for (int64_t i = 0; i < V; ++i) {
        const int32_t b = o->bvm[i];
        if (K[b] >= 2 && c[i] > 0.f && o->av[i] > 0.f) ptr[b + 1]++;
    }
    for (int64_t b = 0; b < B; ++b) ptr[b + 1] += ptr[b];
    cand_t* cs = (cand_t*)malloc(sizeof(cand_t) * (size_t)(ptr[B] > 0 ? ptr[B] : 1));
    int64_t* cur = (int64_t*)malloc(sizeof(int64_t) * (size_t)(B > 0 ? B : 1));
    for (int64_t b = 0; b < B; ++b) cur[b] = ptr[b];
    for (int64_t i = 0; i < V; ++i) {
        const int32_t b = o->bvm[i];
        if (K[b] >= 2 && c[i] > 0.f && o->av[i] > 0.f) { cs[cur[b]].c = c[i]; cs[cur[b]].i = i; cur[b]++; }
    }
    for (int64_t b = 0; b < B; ++b) {
        if (!sel[b]) continue;
        if (K[b] == 1) {                                                  /* :168-169 */
            asg[mi[b]] = sgnf(score[mi[b]]);
            if (trace) trace_push(o, o->iters_done, mi[b], (int64_t)sgnf(score[mi[b]]));
            continue;
        }
        const int64_t n = ptr[b + 1] - ptr[b];
        qsort(cs + ptr[b], (size_t)n, sizeof(cand_t), cand_cmp);
        for (int64_t k = 0; k < n && k < K[b]; ++k) {
            const int64_t i = cs[ptr[b] + k].i;
            asg[i] = sgnf(score[i]);
            if (trace) trace_push(o, o->iters_done, i, (int64_t)sgnf(score[i]));
        }
    }
    free(mi); free(K); free(ptr); free(cs); free(cur);
}

/* stateless form (pdp_decimation_select): problem_sel uint8 [B] or NULL = all; a problem takes part when selected, free
 * of NaN coefficients and with a positive coefficient sum; nav = the oracle's active variables.  Returns 0 or -1. */
int sid_decimation_select(ora_t* o, const float* coeff, const float* score, const uint8_t* problem_sel, float frac, float* out) {
    const int64_t V = o->V, B = o->B;
    if (!valid_fraction(frac) || (o->strict && frac > 0.f)) return -1;
    float* sum = (float*)calloc((size_t)(B > 0 ? B : 1), sizeof(float));
    float* nav = (float*)calloc((size_t)(B > 0 ? B : 1), sizeof(float));
    int* bad = (int*)calloc((size_t)(B > 0 ? B : 1), sizeof(int));
    int* sel = (int*)calloc((size_t)(B > 0 ? B : 1), sizeof(int));
    for (int64_t i = 0; i < V; ++i) {
        const int32_t b = o->bvm[i];
        if (coeff[i] != coeff[i]) bad[b] = 1;
        sum[b] += coeff[i];
        nav[b] += o->av[i];
    }
    for (int64_t b = 0; b < B; ++b) sel[b] = (problem_sel ? problem_sel[b] != 0 : 1) && !bad[b] && sum[b] > 0.f;
    for (int64_t i = 0; i < V; ++i) out[i] = 0.f;
    decimation_rule(o, coeff, score, sel, nav, frac, out, 0);
    free(sum); free(nav); free(bad); free(sel);
    return 0;
}

/* ------------------------------------------------------------------------------------------ */
/* SequentialDecimator.forward with the fraction rule (the oracle's decimate(), pdp_decimate.py:122-177)          */
/* ------------------------------------------------------------------------------------------ */
static void sid_decimate(ora_t* o, float tol, float t_max, int has_active_mask, float pi, float frac) {
    const int64_t E = o->E, V = o->V, B = o->B;
    float* eta = o->tE0;                 /* message_state[1][:, 0] */
    for (int64_t e = 0; e < E; ++e) eta[e] = o->fs2[2 * e];
    if (!o->has_counters) { for (int64_t b = 0; b < B; ++b) o->counters[b] = 0.f; o->has_counters = 1; }

    if (has_active_mask) {               /* :127-133 */
        float* sv = o->tV0; float* mb = o->tB0;
        smooth_max_var(o, eta, sv);
        for (int64_t i = 0; i < V; ++i) sv[i] = sv[i] * o->av[i];
        sparse_max_batch(o, sv, mb);
        for (int64_t b = 0; b < B; ++b) if (mb[b] <= 1e-10f) o->active[b] = 0;
    }

    /* :135 -- `_active_variables.sum() > 0` is batch-global in the reference */
    double nav = 0; for (int64_t i = 0; i < V; ++i) nav += o->av[i];
    float* navb = (float*)malloc(sizeof(float) * (size_t)(B > 0 ? B : 1));   /* (o->tB1 holds `norm` below) */
    for (int64_t b = 0; b < B; ++b) navb[b] = 0.f;
    for (int64_t i = 0; i < V; ++i) navb[o->bvm[i]] += o->av[i];

    if (o->has_prev && (o->strict ? (nav > 0) : 1)) {
        float* d = o->tE1; float* sd = o->tV0; float* db = o->tB0;
        for (int64_t e = 0; e < E; ++e) {
            d[e] = fabsf(o->prev[e] - eta[e]);
            if (o->em_set) d[e] = d[e] * o->em[e];          /* :138-139 */
        }
        smooth_max_var(o, d, sd);
        for (int64_t i = 0; i < V; ++i) sd[i] = sd[i] * o->av[i];
        sparse_max_batch(o, sd, db);
        float* conv = o->tB0;   /* reuse: conv[b] written after db[b] is consumed */
        int* in_block = (int*)malloc(sizeof(int) * (size_t)(B > 0 ? B : 1));
        for (int64_t b = 0; b < B; ++b) {
            in_block[b] = o->strict ? 1 : (navb[b] > 0.f);
            if (!in_block[b]) { conv[b] = 0.f; continue; }
            float v = db[b];
            if (v < tol) o->counters[b] = 0.f;                        /* :145 */
            float c = (v < tol) ? 1.f : 0.f;                          /* :146 */
            if (o->counters[b] >= t_max) { c = 1.f; o->counters[b] = 0.f; }   /* :147-148 */
            conv[b] = c;
        }
        float* convv = o->tV1;
        double nconv = 0;
        for (int64_t i = 0; i < V; ++i) { convv[i] = conv[o->bvm[i]]; nconv += convv[i]; }   /* :150 */
        if (nconv > 0) {                                              /* :152 */
            float* score = o->tV2; float* coeff = o->tV3;
            ora_score(o, o->fs2, o->af, pi, score);
            for (int64_t i = 0; i < V; ++i) coeff[i] = fabsf(score[i]) * o->av[i] * convv[i];
            float* norm = o->tB1;
            for (int64_t b = 0; b < B; ++b) norm[b] = 0.f;
            for (int64_t i = 0; i < V; ++i) norm[o->bvm[i]] += coeff[i];      /* :160 */
            float csum = 0.f; for (int64_t i = 0; i < V; ++i) csum += coeff[i];
            if (o->strict ? (csum > 0.f) : 1) {                       /* :158 */
                float* asg = o->tV0;
                for (int64_t i = 0; i < V; ++i) asg[i] = 0.f;
                int any = 0;
                int* sel = (int*)malloc(sizeof(int) * (size_t)(B > 0 ? B : 1));
                for (int64_t b = 0; b < B; ++b) {
                    if (o->strict) sel[b] = (has_active_mask ? o->active[b] : 1) && (norm[b] != 0.f);
                    else           sel[b] = (has_active_mask ? o->active[b] : 1) && in_block[b] && (norm[b] > 0.f);
                    any |= sel[b];
                }
                decimation_rule(o, coeff, score, sel, navb, frac, asg, 1);   /* :160-169 with the fraction */
                free(sel);
                if (any) ora_set_variables(o, asg);                   /* :171 */
            }
        }
        for (int64_t b = 0; b < B; ++b) if (in_block[b]) o->counters[b] = o->counters[b] + 1.f;   /* :173 */
        free(in_block);
    }
    for (int64_t e = 0; e < E; ++e) o->prev[e] = eta[e];              /* :175 */
    o->has_prev = 1;
    free(navb);
}

/* ------------------------------------------------------------------------------------------ */
/* one trip of the _forward_core loop: solver.py:365-384 + trainer.py:150-162                   */
/* ------------------------------------------------------------------------------------------ */
/* returns the number of still-active problems (or B when there is no termination check) */
int64_t sid_iterate(ora_t* o, float tol, float t_max, int check_termination, int batch_replication, float pi, float frac) {
    const int64_t E = o->E, B = o->B;
    o->iters_done++;
    float* nq = ALLOC(float, 3 * E); float* nf = ALLOC(float, 2 * E);
    float* ft = o->tF1; float* ps = ALLOC(float, o->V); float* ns = ALLOC(float, o->V);
    sp_step_core(o, o->q3, o->fs2, o->em_in_state ? o->em : NULL, o->pq3, o->pfs2,
                 check_termination ? o->active : NULL, pi, nq, nf, o->tE1, o->tE2, ft, ps, ns);
    /* p-d-p: the decimator returns the propagator state unchanged, so both states are the new one */
    memcpy(o->q3, nq, sizeof(float) * 3 * (size_t)E); memcpy(o->fs2, nf, sizeof(float) * 2 * (size_t)E);
    memcpy(o->pq3, nq, sizeof(float) * 3 * (size_t)E); memcpy(o->pfs2, nf, sizeof(float) * 2 * (size_t)E);
    free(nq); free(nf); free(ps); free(ns);

    sid_decimate(o, tol, t_max, check_termination, pi, frac);

    compute_edge_mask(o);                                             /* solver.py:370-371 */
    double s = 0; for (int64_t e = 0; e < E; ++e) s += o->em[e];
    o->em_in_state = (s < (double)E);                                 /* solver.py:373-374 */

    if (!check_termination) return B;
    /* predictor (IdentityPredictor) + _update_solution leave _solution unchanged; trainer.py:150-162 */
    float* solved = ALLOC(float, B); float* nun = ALLOC(float, B);
    ora_cnf_eval(o, o->sol, solved, nun);
    if (batch_replication > 1) {
        const int64_t B0 = B / batch_replication;
        for (int64_t j = 0; j < B0; ++j) {
            float any = 0.f;
            for (int r = 0; r < batch_replication; ++r) any += (solved[r * B0 + j] > 0.5f) ? 1.f : 0.f;
            for (int r = 0; r < batch_replication; ++r)
                if (o->active[r * B0 + j]) o->active[r * B0 + j] = (any == 0.f) ? 1 : 0;
        }
    } else {
        for (int64_t b = 0; b < B; ++b) if (o->active[b]) o->active[b] = (solved[b] <= 0.5f) ? 1 : 0;
    }
    free(solved); free(nun);
    int64_t na = 0; for (int64_t b = 0; b < B; ++b) na += o->active[b];
    return na;
}

/* solver.py:355-386: runs up to T iterations, returns the number executed */
int64_t sid_run(ora_t* o, int64_t T, float tol, float t_max, int check_termination, int batch_replication, float pi, float frac) {
    int64_t t = 0;
    for (; t < T; ++t) {
        int64_t na = sid_iterate(o, tol, t_max, check_termination, batch_replication, pi, frac);
        if (check_termination && na <= 0) { ++t; break; }
    }
    return t;
}
