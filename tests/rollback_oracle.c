/*
 * TEST INFRASTRUCTURE ONLY -- CPU restatement of conflict rollback for SP-inspired decimation (include/pdp_b200.h,
 * pdp_set_conflict_rollback) on top of tests/sid_oracle.c, included as it is.  What differs is the decimator and the loop
 * that calls it: rb_decimate restates sid_decimate with the step size K_b = max(1, floor((double)f * A_b) >> h_b) and the
 * rollback of a K_b >= 2 step that ends in a unit-propagation conflict; rb_iterate / rb_run restate sid_iterate / sid_run
 * around it.  With rollback off every function below computes what its sid_oracle.c counterpart computes.  Defined for
 * strict = 0.  The oracle keeps no conflict flag: a problem has conflicted iff its is_sat is 0, which the oracle writes only
 * on a conflict (solver.py:245), as the library writes PDP_FLAG_UP_CONFLICT together with is_sat = 0.
 */
#include "sid_oracle.c"

typedef struct {
    int64_t B;
    int on;                  /* rollback on (pdp_set_conflict_rollback with a buffer)            */
    int64_t *h, *r, *last;   /* [B] halving exponent, rollback count, iteration of the last one  */
} rb_t;

rb_t* rb_create(const ora_t* o) {
    rb_t* rb = ALLOC(rb_t, 1);
    rb->B = o->B;
    rb->h = ALLOC(int64_t, o->B); rb->r = ALLOC(int64_t, o->B); rb->last = ALLOC(int64_t, o->B);
    return rb;
}
void rb_destroy(rb_t* rb) {
    if (!rb) return;
    free(rb->h); free(rb->r); free(rb->last); free(rb);
}
void rb_set(rb_t* rb, int on) { rb->on = on; }
void rb_get(const rb_t* rb, int64_t* h, int64_t* r, int64_t* last) {
    memcpy(h, rb->h, sizeof(int64_t) * (size_t)rb->B);
    memcpy(r, rb->r, sizeof(int64_t) * (size_t)rb->B);
    memcpy(last, rb->last, sizeof(int64_t) * (size_t)rb->B);
}

/* K_b with the halving exponent (h = 0: sel_k) */
static int64_t rb_k(float f, float nav, int64_t h) {
    const int64_t k = (int64_t)floor((double)f * (double)nav);
    const int64_t q = k >> (h < 62 ? h : 62);
    return q < 1 ? 1 : q;
}

/* decimation_rule with K_b = rb_k(frac, nav[b], h[b]) (h NULL: every h_b = 0); K [B] receives K_b (0: not selected) */
static void rb_rule(ora_t* o, const float* c, const float* score, const int* sel, const float* nav, float frac,
                    const int64_t* h, float* asg, int64_t* K) {
    const int64_t V = o->V, B = o->B;
    int64_t* mi = (int64_t*)malloc(sizeof(int64_t) * (size_t)(B > 0 ? B : 1));
    int64_t* ptr = (int64_t*)calloc((size_t)(B + 1), sizeof(int64_t));
    sparse_argmax_batch(o, c, mi);
    for (int64_t b = 0; b < B; ++b) K[b] = sel[b] ? rb_k(frac, nav[b], h ? h[b] : 0) : 0;
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
            trace_push(o, o->iters_done, mi[b], (int64_t)sgnf(score[mi[b]]));
            continue;
        }
        const int64_t n = ptr[b + 1] - ptr[b];
        qsort(cs + ptr[b], (size_t)n, sizeof(cand_t), cand_cmp);
        for (int64_t k = 0; k < n && k < K[b]; ++k) {
            const int64_t i = cs[ptr[b] + k].i;
            asg[i] = sgnf(score[i]);
            trace_push(o, o->iters_done, i, (int64_t)sgnf(score[i]));
        }
    }
    free(mi); free(ptr); free(cs); free(cur);
}

/* ora_set_variables (fix + UP + peel closure) with the rollback: a problem that took K_b >= 2 variables, had not conflicted
 * before and has now gets its av / af / sol / is_sat from before the fix back, and h_b, r_b grow by one */
static void rb_set_variables(ora_t* o, rb_t* rb, const float* asg, const int64_t* K) {
    const int64_t V = o->V, F = o->F, B = o->B;
    float* av0 = ALLOC(float, V); float* af0 = ALLOC(float, F); float* sol0 = ALLOC(float, V); float* sat0 = ALLOC(float, B);
    memcpy(av0, o->av, sizeof(float) * (size_t)V); memcpy(af0, o->af, sizeof(float) * (size_t)F);
    memcpy(sol0, o->sol, sizeof(float) * (size_t)V); memcpy(sat0, o->is_sat, sizeof(float) * (size_t)B);
    ora_set_variables(o, asg);
    if (rb->on) {
        int* roll = ALLOC(int, B);
        for (int64_t b = 0; b < B; ++b) roll[b] = K[b] >= 2 && sat0[b] != 0.f && o->is_sat[b] == 0.f;
        for (int64_t i = 0; i < V; ++i) if (roll[o->bvm[i]]) { o->av[i] = av0[i]; o->sol[i] = sol0[i]; }
        for (int64_t a = 0; a < F; ++a) if (roll[o->bfm[a]]) o->af[a] = af0[a];
        for (int64_t b = 0; b < B; ++b)
            if (roll[b]) { o->is_sat[b] = sat0[b]; rb->h[b]++; rb->r[b]++; rb->last[b] = o->iters_done; }
        free(roll);
    }
    free(av0); free(af0); free(sol0); free(sat0);
}

/* sid_decimate with rb_rule and rb_set_variables */
static void rb_decimate(ora_t* o, rb_t* rb, float tol, float t_max, int has_active_mask, float pi, float frac) {
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

    float* navb = (float*)malloc(sizeof(float) * (size_t)(B > 0 ? B : 1));
    for (int64_t b = 0; b < B; ++b) navb[b] = 0.f;
    for (int64_t i = 0; i < V; ++i) navb[o->bvm[i]] += o->av[i];

    if (o->has_prev) {                   /* :135, strict = 0 */
        float* d = o->tE1; float* sd = o->tV0; float* db = o->tB0;
        for (int64_t e = 0; e < E; ++e) {
            d[e] = fabsf(o->prev[e] - eta[e]);
            if (o->em_set) d[e] = d[e] * o->em[e];          /* :138-139 */
        }
        smooth_max_var(o, d, sd);
        for (int64_t i = 0; i < V; ++i) sd[i] = sd[i] * o->av[i];
        sparse_max_batch(o, sd, db);
        float* conv = o->tB0;
        int* in_block = (int*)malloc(sizeof(int) * (size_t)(B > 0 ? B : 1));
        for (int64_t b = 0; b < B; ++b) {
            in_block[b] = navb[b] > 0.f;
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
            /* the assignment gets its own buffer: ora_set_variables copies it into tV3 (= coeff) */
            float* asg = ALLOC(float, V);
            int64_t* K = ALLOC(int64_t, B);
            int any = 0;
            int* sel = (int*)malloc(sizeof(int) * (size_t)(B > 0 ? B : 1));
            for (int64_t b = 0; b < B; ++b) {
                sel[b] = (has_active_mask ? o->active[b] : 1) && in_block[b] && (norm[b] > 0.f);
                any |= sel[b];
            }
            rb_rule(o, coeff, score, sel, navb, frac, rb->on ? rb->h : NULL, asg, K);   /* :160-169 */
            if (any) rb_set_variables(o, rb, asg, K);                 /* :171 + rollback */
            free(sel); free(asg); free(K);
        }
        for (int64_t b = 0; b < B; ++b) if (in_block[b]) o->counters[b] = o->counters[b] + 1.f;   /* :173 */
        free(in_block);
    }
    for (int64_t e = 0; e < E; ++e) o->prev[e] = eta[e];              /* :175 */
    o->has_prev = 1;
    free(navb);
}

/* sid_iterate with rb_decimate */
int64_t rb_iterate(ora_t* o, rb_t* rb, float tol, float t_max, int check_termination, int batch_replication, float pi,
                   float frac) {
    const int64_t E = o->E, B = o->B;
    o->iters_done++;
    float* nq = ALLOC(float, 3 * E); float* nf = ALLOC(float, 2 * E);
    float* ft = o->tF1; float* ps = ALLOC(float, o->V); float* ns = ALLOC(float, o->V);
    sp_step_core(o, o->q3, o->fs2, o->em_in_state ? o->em : NULL, o->pq3, o->pfs2,
                 check_termination ? o->active : NULL, pi, nq, nf, o->tE1, o->tE2, ft, ps, ns);
    memcpy(o->q3, nq, sizeof(float) * 3 * (size_t)E); memcpy(o->fs2, nf, sizeof(float) * 2 * (size_t)E);
    memcpy(o->pq3, nq, sizeof(float) * 3 * (size_t)E); memcpy(o->pfs2, nf, sizeof(float) * 2 * (size_t)E);
    free(nq); free(nf); free(ps); free(ns);

    rb_decimate(o, rb, tol, t_max, check_termination, pi, frac);

    compute_edge_mask(o);                                             /* solver.py:370-371 */
    double s = 0; for (int64_t e = 0; e < E; ++e) s += o->em[e];
    o->em_in_state = (s < (double)E);                                 /* solver.py:373-374 */

    if (!check_termination) return B;
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

int64_t rb_run(ora_t* o, rb_t* rb, int64_t T, float tol, float t_max, int check_termination, int batch_replication,
               float pi, float frac) {
    int64_t t = 0;
    for (; t < T; ++t) {
        int64_t na = rb_iterate(o, rb, tol, t_max, check_termination, batch_replication, pi, frac);
        if (check_termination && na <= 0) { ++t; break; }
    }
    return t;
}
