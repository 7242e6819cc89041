// pdp_loop.cu -- the persistent cooperative kernels: the whole propagate -> decimate -> predict loop of
// the p-d-p model (reference pdp/nn/solver.py:355-386) runs inside ONE launch with grid-wide barriers
// between its phases, per-problem convergence / termination flags, and no host round trip.
// The reference needs >= 6 device->host synchronisations per iteration for the same control flow.
#include "pdp_device.cuh"

namespace {

// ------------------------------------------------------------------------------------------------
// SequentialDecimator decisions, one thread per problem (pdp_decimate.py:127-150,173)
// ------------------------------------------------------------------------------------------------
__device__ __forceinline__ void decide_phase(const KArgs& A, int iter, const pdp_sp_params& prm, bool has_prev, bool local_ok,
                                             bool blocked) {
    const pdp_state& s = A.s;
    const int slot = CTRL_CONV + (iter & 1);
    WARP_STRIDED(b, A.g.B) {
        if (b >= A.g.B) continue;
        uint8_t cv = 0;
        bool near = false;       // close to the convergence test: worth scoring inside the next variable pass
        // a NaN produced during this iteration's passes puts the problem on the sticky-NaN path from
        // the next iteration on (no old NaN existed while it was produced)
        if (s.nanpend[b]) { s.nanpend[b] = 0; s.nanflag[b] = 1; s.ctrl[CTRL_ANY_NAN] = 1; }
        if (s.active[b]) {
            const uint32_t nanb = s.st_nan[b];
            const uint32_t mx0 = s.st_max[2 * b], mn0 = s.st_min[2 * b];
            const uint32_t mx1 = s.st_max[2 * b + 1], mn1 = s.st_min[2 * b + 1];
            const bool seen0 = (mn0 != 0x7f800000u) || (mx0 != 0u);
            bool act = true;
            if (prm.check_termination) {
                // util.sparse_max over an empty column gives 0 + min - 1
                float M = (nanb & 1u) ? __int_as_float(0x7fc00000) : (seen0 ? sparse_max_round(u2f(mx0), u2f(mn0)) : -1.f);
                if (M <= 1e-10f) {   // pdp_decimate.py:133
                    s.active[b] = 0; act = false;
                    s.flags[b] |= PDP_FLAG_TRIVIAL;
                    s.freeze_iter[b] = iter;
                    atomicSub(&s.ctrl[CTRL_NUM_ACTIVE], 1);
                }
            }
            if (has_prev && s.nav[b] > 0) {   // pdp_decimate.py:135
                const bool seen1 = (mn1 != 0x7f800000u) || (mx1 != 0u);
                float D = (nanb & 2u) ? __int_as_float(0x7fc00000) : (seen1 ? sparse_max_round(u2f(mx1), u2f(mn1)) : -1.f);
                int cnt = s.counters[b];
                if (D < prm.tolerance) cnt = 0;                    // :145
                bool c = D < prm.tolerance;                         // :146
                if (cnt >= prm.t_max) { c = true; cnt = 0; }        // :147-148
                cv = (c && act) ? 1 : 0;
                s.counters[b] = cnt + 1;                            // :173
                // will it converge in the NEXT iteration?  It just did (decimation keeps the surveys converged), its counter
                // runs out, or the statistic, which decays geometrically, extrapolates below the tolerance
                const float Dp = s.last_d[b];
                s.last_d[b] = D;
                near = act && (c || cnt + 1 >= prm.t_max || (Dp > 0.f && D < Dp && D * (D / Dp) < 1.25f * prm.tolerance));
            }
            if (nanb) s.flags[b] |= PDP_FLAG_CONTRADICTION;
            s.st_max[2 * b] = 0u; s.st_max[2 * b + 1] = 0u;
            s.st_min[2 * b] = 0x7f800000u; s.st_min[2 * b + 1] = 0x7f800000u;
            s.st_nan[b] = 0u; s.nav[b] = 0;
        }
        s.conv[b] = cv;
        // scores of this iteration's variable pass are valid if it was asked for them and ran blocked
        s.have_score[b] = (blocked && s.want_score[b]) ? 1 : 0;
        s.want_score[b] = (near && !s.nanflag[b] && (!local_ok || !loc_problem_is_small(A.g, (int)b))) ? 1 : 0;
        if (cv) {
            s.ctrl[slot] = 1;
            if (!local_ok || !loc_problem_is_small(A.g, (int)b)) s.ctrl[CTRL_CONVBIG + (iter & 1)] = 1;
            else s.loc_list[atomicAdd(&s.ctrl[CTRL_LOC_COUNT], 1)] = (int32_t)b;
        }
    }
}

// pdp_decimate.py:158-171: fix the arg-max variable of every converged, still active problem
__device__ __forceinline__ void select_and_fix_phase(const KArgs& A, int iter, bool frontier) {
    const pdp_graph& g = A.g; const pdp_state& s = A.s;
    const int slot = CTRL_FIX + (iter & 1);
    const ListQueue q = frontier_queue(s);
    // warp per problem: every lane takes the same decisions, the fix itself is spread over the lanes
    for (int64_t b = gwarp(); b < g.B; b += gwarps()) {
        if (!s.conv[b]) continue;
        if (!s.c_nan[b] && u2f(s.c_max[b]) > 0.f && s.arg_idx[b] != 0x7fffffff) {
            const int i = s.arg_idx[b];
            const float sg = sgnf(s.score[i]);
            if (sg != 0.f && s.av[i]) {
                __syncwarp();     // everybody has read av[i] before lane 0 clears it
                if (frontier) fix_variable<32>(g, s, i, sg, q);
                else fix_variable<32>(g, s, i, sg);
                if (lane_id() == 0) {
                    s.masked[b] = 1; s.dirty[b] = 1;
                    s.ctrl[slot] = 1; s.ctrl[CTRL_ANY_DIRTY] = 1;
                    record_fix(A, iter, i, sg);
                }
            }
        }
        __syncwarp();             // ... and the per-problem arg-max state before lane 0 resets it
        if (lane_id() == 0) { s.c_max[b] = 0u; s.c_min[b] = 0x7f800000u; s.c_nan[b] = 0u; s.arg_idx[b] = 0x7fffffff; }
    }
}

// the fix step of the fused loop with a fraction: the arg-max fixes (K_b == 1) and the top-K fixes of the other problems,
// one warp per taken variable (fix_variable<32>, + the frontier lists).  Fixes of one step commute: a clause is
// de-activated iff it holds a newly true literal (_set_variable_core, solver.py:205-226).
__device__ __forceinline__ void frac_select_and_fix(const KArgs& A, cg::grid_group& grid, int iter, bool frontier) {
    const pdp_graph& g = A.g; const pdp_state& s = A.s;
    const bool rb = A.rb.av != nullptr;
    sel_grid(A, grid, CoefScore{s}, A.dec_fraction, rb);
    if (rb) rb_snapshot_grid(A);
    select_and_fix_phase(A, iter, frontier);
    if (rb) grid.sync();   // the snapshots are complete before the top-K fixes
    const int slot = CTRL_FIX + (iter & 1);
    const ListQueue q = frontier_queue(s);
    for (int64_t base = gwarp() * 32; base < g.V; base += gwarps() * 32) {
        const int64_t i = base + lane_id();
        bool take = false;
        float sg = 0.f;
        if (i < g.V) {
            const int b = g.bvm[i];
            if (s.sel_need[b] == 0) {
                take = sel_taken(s, b, i, fabsf(s.score[i]) * (float)s.av[i], s.av[i] != 0);
                sg = sgnf(s.score[i]);
            }
        }
        unsigned m = __ballot_sync(0xffffffffu, take);
        while (m) {
            const int src = __ffs(m) - 1;
            m &= m - 1;
            const int vi = (int)__shfl_sync(0xffffffffu, i, src);
            const float vsg = __shfl_sync(0xffffffffu, sg, src);
            if (frontier) fix_variable<32>(g, s, vi, vsg, q);
            else fix_variable<32>(g, s, vi, vsg);
            if (lane_id() == 0) {
                const int b = g.bvm[vi];
                s.masked[b] = 1; s.dirty[b] = 1;
                s.ctrl[slot] = 1; s.ctrl[CTRL_ANY_DIRTY] = 1;
                record_fix(A, iter, vi, vsg);
            }
            __syncwarp();
        }
    }
}

// trainer.py:150-162 on the dirty problems
__device__ __forceinline__ void termination_phase(const KArgs& A, int iter, int rep) {
    const pdp_graph& g = A.g; const pdp_state& s = A.s;
    const int64_t B0 = g.B / rep;
    WARP_STRIDED(j, B0) {
        if (j >= B0) continue;
        bool any = false;
        for (int r = 0; r < rep; ++r) {
            const int64_t b = (int64_t)r * B0 + j;
            if (s.dirty[b] && s.n_unsat[b] == 0) any = true;
        }
        for (int r = 0; r < rep; ++r) {
            const int64_t b = (int64_t)r * B0 + j;
            if (any && s.active[b]) {
                s.active[b] = 0;
                s.freeze_iter[b] = iter;
                atomicSub(&s.ctrl[CTRL_NUM_ACTIVE], 1);
            }
            if (s.dirty[b] && s.n_unsat[b] == 0) s.flags[b] |= PDP_FLAG_SOLVED;
            s.dirty[b] = 0; s.n_unsat[b] = 0;
        }
    }
    if (gtid() == 0) s.ctrl[CTRL_ANY_DIRTY] = 0;
}

// FAST: the blocked shared-memory passes (pi == 0, q_u only); otherwise the generic passes.
// FRAC: a decimation fraction is set (pdp_set_decimation_fraction); a separate instance, so that the top-K selection
// takes nothing from the registers of the instance the reference's rule runs in
template <bool FAST, bool FULL, int CTAS, bool FRAC>
__global__ void __launch_bounds__(FAST ? SweepCfg<CTAS>::kThreads : 256, FAST ? CTAS : 1)
k_sp_run(const __grid_constant__ KArgs A, const __grid_constant__ pdp_sp_params prm, int32_t* d_iters_done) {
    extern __shared__ __align__(128) unsigned char smem_dyn[];
    cg::grid_group grid = cg::this_grid();
    const pdp_state& s = A.s;
    int iter = s.ctrl[CTRL_ITER];
    bool has_prev = s.ctrl[CTRL_HAS_PREV] != 0;
    bool use_mask = s.ctrl[CTRL_USE_MASK] != 0;
    bool em_set = s.ctrl[CTRL_EM_SET] != 0;
    int gen_left = FAST ? s.ctrl[CTRL_GEN_ITERS] : 0;
    const int rep = prm.batch_replication > 1 ? prm.batch_replication : 1;
    const bool local_ok = A.g.contiguous_problems && rep == 1 && !(prm.flags & 2);
    const bool frontier = s.ctrl[CTRL_CLOSED] != 0 && !(prm.flags & 4);   // flags bit 2: full-scan closure (A/B, tests)
    int executed = 0;
    int sm_rank = 0;
    // completion barrier of the blocked passes' bulk copies: one mbarrier for the kernel's lifetime (static shared memory:
    // the CTA-local decimation borrows the dynamic part)
    __shared__ __align__(8) uint64_t sm_bulk_bar;
    BulkBar bb{&sm_bulk_bar, 0u};
    if (FAST) {
        if (threadIdx.x == 0) mbar_init(&sm_bulk_bar, 1);
        __syncthreads();
    }
    if (FAST && CTAS == 2) {   // rank of this CTA among the CTAs of its SM (the counters are zeroed before the launch)
        __shared__ int sm_rank_s;
        if (threadIdx.x == 0) {
            unsigned smid;
            asm volatile("mov.u32 %0, %%smid;" : "=r"(smid));
            sm_rank_s = atomicAdd(&s.sm_ctr[smid % PDP_MAX_SMS], 1) & 1;
        }
        __syncthreads();
        sm_rank = sm_rank_s;
    }
    if (gtid() == 0) { s.ctrl[CTRL_NEXT_CBLK] = 0; s.ctrl[CTRL_NEXT_VBLK] = 0; s.ctrl[CTRL_LOC_COUNT] = 0; s.ctrl[CTRL_LOC_NEXT] = 0; }
#ifdef PDP_PHASE_TIMING
#define GRID_SYNC() do { const long long _g0 = clock64(); grid.sync(); if (threadIdx.x == 0 && A.trace) atomicAdd(&A.trace[7], (int)((clock64() - _g0) >> 10)); } while (0)
#else
#define GRID_SYNC() grid.sync()
#endif
#ifdef PDP_PHASE_TIMING
    const long long _kernel_t0 = clock64();
#endif
    grid.sync();   // everybody has read the control block before anyone may change it
#ifdef PDP_PHASE_TIMING
    long long _lt = clock64();
#define LOOP_T(slot_) do { if (threadIdx.x == 0 && A.trace) { const long long _n = clock64(); atomicAdd(&A.trace[slot_], (int)((_n - _lt) >> 10)); _lt = _n; } } while (0)
#else
#define LOOP_T(slot_) do {} while (0)
#endif
    for (int it = 0; it < prm.iterations; ++it) {
        ++iter;
        const int r = (iter - 1) & 1, w = iter & 1;
        LOOP_T(23);
        const bool blocked = FAST && gen_left <= 0;
        if (gen_left > 0) --gen_left;
        // ---- propagate, clause side: eta(t) from q(t-1)   (pdp_propagate.py:161-175)
        if (blocked) {
            blk_clause_pass<CTAS>(A, r, use_mask, smem_dyn, sm_rank, bb);
        } else {
            gen_clause_side<GEN_ALL>(A, r, use_mask);
        }
        LOOP_T(16);
        if (gtid() == 0) { s.ctrl[CTRL_NEXT_VBLK] = 0; s.ctrl[CTRL_LOC_COUNT] = 0; s.ctrl[CTRL_LOC_NEXT] = 0; }
        if (gtid() == 0) { s.ctrl[CTRL_CONV + ((iter + 1) & 1)] = 0; s.ctrl[CTRL_FIX + ((iter + 1) & 1)] = 0; s.ctrl[CTRL_CONVBIG + ((iter + 1) & 1)] = 0; }
        GRID_SYNC();
        LOOP_T(17);
        // ---- propagate, variable side: q(t) from eta(t-1) (pdp_propagate.py:184-218), fused with the
        //      decimator statistics of eta(t) against eta(t-1) (pdp_decimate.py:127-143)
        if (blocked) {
            blk_var_pass<CTAS>(A, r, use_mask, has_prev, em_set, smem_dyn, sm_rank, bb);
        } else {
            gen_var_side<GEN_ALL, FULL>(A, r, use_mask, prm.pi);
            gen_stats<GEN_ALL>(A, w, has_prev, em_set);
        }
        LOOP_T(18);
        GRID_SYNC();
        if (gtid() == 0) s.ctrl[CTRL_NEXT_CBLK] = 0;   // the variable pass is over; the next clause pass is a barrier away
        LOOP_T(19);
        // ---- decimate: decisions -> (score, argmax, fix, simplify)
        decide_phase(A, iter, prm, has_prev, local_ok, blocked);
        GRID_SYNC();
        LOOP_T(20);
        if (local_ok && s.ctrl[CTRL_CONV + (iter & 1)]) {
            // converged problems one CTA can walk: scoring, arg-max, fix, closure, CNF check, termination, CTA-local
            loc_decimate_all<FRAC>(A, iter, w, prm.pi, prm.check_termination != 0, FAST ? smem_dyn : nullptr,
                                   FAST ? SweepCfg<CTAS>::kSmem : 0);
            LOOP_T(21);
            GRID_SYNC();
            LOOP_T(22);
        }
        if (s.ctrl[local_ok ? (CTRL_CONVBIG + (iter & 1)) : (CTRL_CONV + (iter & 1))]) {
            LOOP_T(23);
            score_phase(A, w, prm.pi);
            GRID_SYNC();
            LOOP_T(24);
            argmax_phase(A, CoefScore{s});
            GRID_SYNC();
            if (FRAC) frac_select_and_fix(A, grid, iter, frontier);
            else select_and_fix_phase(A, iter, frontier);
            GRID_SYNC();
            LOOP_T(25);
            if (s.ctrl[CTRL_FIX + (iter & 1)]) {
                if (frontier) closure_frontier<FRAC>(A, grid);
                else closure<FRAC>(A, grid);
            }
            if (FRAC && s.ctrl[CTRL_RB]) {   // conflict rollback: some top-K step ended in a conflict
                rb_restore_grid(A, iter);
                GRID_SYNC();
                if (gtid() == 0) s.ctrl[CTRL_RB] = 0;   // (read by everybody before the barrier)
            }
            LOOP_T(26);
        }
        has_prev = true;   // pdp_decimate.py:175
        em_set = true;     // solver.py:370-371
        use_mask = true;   // solver.py:373-374 (multiplying by an all-ones mask is the identity)
        ++executed;
        // ---- predict + termination: IdentityPredictor/_update_solution leave _solution as is
        if (prm.check_termination) {
            if (s.ctrl[CTRL_ANY_DIRTY] && !(prm.flags & 8)) {   // flags bit 3: the caller runs its own termination check
                LOOP_T(23);
                cnf_count_dirty(A);
                GRID_SYNC();
                LOOP_T(27);
                termination_phase(A, iter, rep);
                GRID_SYNC();
                LOOP_T(28);
            }
            if (s.ctrl[CTRL_NUM_ACTIVE] <= 0) break;
        }
    }
    GRID_SYNC();
#ifdef PDP_PHASE_TIMING
    if (threadIdx.x == 0 && A.trace) atomicAdd(&A.trace[6], (int)((clock64() - _kernel_t0) >> 10));
#endif
    if (gtid() == 0) {
        s.ctrl[CTRL_ITER] = iter; s.ctrl[CTRL_HAS_PREV] = has_prev; s.ctrl[CTRL_USE_MASK] = use_mask;
        s.ctrl[CTRL_EM_SET] = em_set; s.ctrl[CTRL_ITERS_THIS_RUN] = executed;
        if (FAST) s.ctrl[CTRL_GEN_ITERS] = gen_left;
        if (d_iters_done) *d_iters_done = executed;
    }
}

// SATProblem.simplify on every problem (solver.py:281-285).  (256, 4): coop_blocks launches at most 4 CTAs per SM
__global__ void __launch_bounds__(256, 4) k_simplify(const __grid_constant__ KArgs A) {
    cg::grid_group grid = cg::this_grid();
    const pdp_state& s = A.s;
    WARP_STRIDED(b, A.g.B) { if (b < A.g.B) s.dirty[b] = 1; }
    if (gtid() == 0) s.ctrl[CTRL_ANY_DIRTY] = 1;
    grid.sync();
    closure(A, grid);
    if (gtid() == 0) s.ctrl[CTRL_CLOSED] = 1;   // every problem was dirty: all of them are closed now
}

// SATProblem.set_variables (solver.py:275-279): assignment [V] float in {-1,0,1}
__global__ void __launch_bounds__(256, 4) k_set_variables(const __grid_constant__ KArgs A, const float* __restrict__ asg) {
    cg::grid_group grid = cg::this_grid();
    const pdp_graph& g = A.g; const pdp_state& s = A.s;
    WARP_STRIDED(b, g.B) { if (b < g.B) s.dirty[b] = 1; }
    if (gtid() == 0) s.ctrl[CTRL_ANY_DIRTY] = 1;
    WARP_STRIDED(i, g.V) {
        if (i >= g.V) continue;
        const float a = asg[i] * (float)s.av[i];   // solver.py:210
        if (fabsf(a) == 1.f) { fix_variable(g, s, (int)i, a); s.masked[g.bvm[i]] = 1; }
    }
    grid.sync();
    closure(A, grid);
    if (gtid() == 0) s.ctrl[CTRL_CLOSED] = 1;
}

// pdp_decimation_select: the decimation rule on caller-supplied coefficients, with the phases of the fused loop
__global__ void __launch_bounds__(256) k_decimation_select(const __grid_constant__ KArgs A, const float* __restrict__ coeff,
                                                           const float* __restrict__ score, const uint8_t* __restrict__ psel,
                                                           float* __restrict__ out) {
    cg::grid_group grid = cg::this_grid();
    const pdp_graph& g = A.g; const pdp_state& s = A.s;
    WARP_STRIDED(i, g.V) { if (i < g.V) out[i] = 0.f; }
    WARP_STRIDED(b, g.B) { if (b < g.B) s.conv[b] = psel ? (psel[b] != 0) : 1; }
    grid.sync();
    KeyedReducer<CoefAcc> red;   // per-problem max / min / NaN of the coefficients (score_phase's statistics)
    WARP_STRIDED(i, g.V) {
        if (i >= g.V) continue;
        const int b = g.bvm[i];
        if (!s.conv[b]) continue;
        red.touch(s, b);
        red.acc.add(coeff[i]);
    }
    red.finish(s);
    grid.sync();
    argmax_phase(A, CoefGiven{coeff});
    grid.sync();
    if (A.dec_fraction > 0.f) sel_grid(A, grid, CoefGiven{coeff}, A.dec_fraction, false);
    WARP_STRIDED(i, g.V) {
        if (i >= g.V) continue;
        const int b = g.bvm[i];
        if (A.dec_fraction > 0.f && s.sel_need[b] == 0 && sel_taken(s, b, i, coeff[i], s.av[i] != 0)) out[i] = sgnf(score[i]);
    }
    WARP_STRIDED(b, g.B) {
        if (b >= g.B) continue;
        if (s.conv[b] && !s.c_nan[b] && u2f(s.c_max[b]) > 0.f && s.arg_idx[b] != 0x7fffffff) out[s.arg_idx[b]] = sgnf(score[s.arg_idx[b]]);
    }
    grid.sync();
    WARP_STRIDED(b, g.B) {   // the per-iteration scratch of the fused loop back to its resting state
        if (b >= g.B) continue;
        s.conv[b] = 0; s.c_max[b] = 0u; s.c_min[b] = 0x7f800000u; s.c_nan[b] = 0u; s.arg_idx[b] = 0x7fffffff; s.sel_need[b] = -1;
    }
}

// pdp_debug_check_edge_mask: edges whose mask bit disagrees with the node masks, per layout
__global__ void __launch_bounds__(256) k_check_edge_mask(const __grid_constant__ KArgs A, int32_t* errs) {
    const pdp_graph& g = A.g; const pdp_state& s = A.s;
    WARP_STRIDED(i, g.V) {
        if (i >= g.V) continue;
        for (int p = g.var_ptr[i]; p < g.var_ptr[i + 1]; ++p) {
            const bool masked = !(s.av[i] && s.af[g.v_cls[p]]);
            if (mbit(g.vmask, g.p_vpos[p]) != masked) atomicAdd(&errs[0], 1);
            if (mbit(g.qmask, g.p_qpos[p]) != masked) atomicAdd(&errs[1], 1);
        }
    }
}

template <typename K>
int coop_blocks(pdp_ctx* ctx, K kernel) {
    int per_sm = 0;
    if (cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, kernel, 256, 0) != cudaSuccess || per_sm < 1) return -1;
    if (per_sm > 4) per_sm = 4;   // 4 x 256 threads per SM: enough bytes in flight, cheap grid barriers
    return per_sm * ctx->num_sms;
}

}  // namespace

// optional decimation trace of ONE context (tests): the buffer belongs to the caller, the context only keeps the pointer
extern "C" int pdp_set_trace_buffer(pdp_ctx* ctx, int32_t* d_trace, int32_t capacity_events) {
    if (!ctx) { pdp_set_error("pdp_set_trace_buffer: null context"); return PDP_ERR_ARG; }
    ctx->trace = d_trace; ctx->trace_cap = d_trace ? capacity_events : 0;
    return PDP_OK;
}

// default start offsets (cycles) of the second CTA of an SM, see blk_stagger (pdp_sweep.cuh); tunable through
// PDP_B200_STAGGER_C / PDP_B200_STAGGER_V for experiments
#ifndef PDP_STAGGER_C
#define PDP_STAGGER_C 0
#endif
#ifndef PDP_STAGGER_V
#define PDP_STAGGER_V 0
#endif
// the snapshot buffer of the conflict rollback: sol [V], is_sat [B] (fp32), av [V], af [F] (bytes)
struct RbLayout { size_t is_sat, av, af, total; };
static RbLayout rb_layout(int64_t V, int64_t F, int64_t B) {
    auto up = [](int64_t x) { return ((size_t)(x > 0 ? x : 0) + 255) & ~(size_t)255; };
    RbLayout l;
    l.is_sat = up(4 * V); l.av = l.is_sat + up(4 * B); l.af = l.av + up(V); l.total = l.af + up(F);
    return l;
}

static KArgs make_args(pdp_ctx* ctx) {
    KArgs A;
    A.g = ctx->g; A.s = ctx->s; A.trace = ctx->trace; A.trace_cap = ctx->trace_cap;
    A.stagger_c = PDP_STAGGER_C; A.stagger_v = PDP_STAGGER_V;
    A.dec_fraction = ctx->dec_fraction;
    A.rb.sol = nullptr; A.rb.is_sat = nullptr; A.rb.av = nullptr; A.rb.af = nullptr;
    if (ctx->rb_scratch) {
        const RbLayout l = rb_layout(ctx->g.V, ctx->g.F, ctx->g.B);
        unsigned char* base = (unsigned char*)ctx->rb_scratch;
        A.rb.sol = (float*)base; A.rb.is_sat = (float*)(base + l.is_sat);
        A.rb.av = base + l.av; A.rb.af = base + l.af;
    }
    if (const char* e = getenv("PDP_B200_STAGGER_C")) A.stagger_c = atoi(e);
    if (const char* e = getenv("PDP_B200_STAGGER_V")) A.stagger_v = atoi(e);
    return A;
}

extern "C" int pdp_sp_run(pdp_ctx* ctx, const pdp_sp_params* params, int32_t* d_iters_done, void* stream_) {
    if (!ctx || !params) { pdp_set_error("pdp_sp_run: null argument"); return PDP_ERR_ARG; }
    if (params->iterations < 0 || params->t_max < 0 || params->batch_replication < 0) { pdp_set_error("pdp_sp_run: negative parameter"); return PDP_ERR_ARG; }
    const int rep = params->batch_replication > 1 ? params->batch_replication : 1;
    if (ctx->g.B % rep != 0) { pdp_set_error("pdp_sp_run: batch size %lld not divisible by replication %d", (long long)ctx->g.B, rep); return PDP_ERR_ARG; }
    cudaStream_t stream = (cudaStream_t)stream_;
    KArgs A = make_args(ctx);
    pdp_sp_params prm = *params;
    ctx->full_state_tracked = prm.full_state ? 1 : 0;
    ctx->last_pi = prm.pi;
    void* args[] = {&A, &prm, &d_iters_done};
    const bool frac = ctx->dec_fraction > 0.f;
    const bool fast = ctx->g.blocked_ok && !prm.full_state && prm.pi == 0.f && !(prm.flags & 1);
    if (fast) {
        // one or two CTAs per SM holding the whole shared memory: co-residency of the cooperative grid is guaranteed
        const int two = (ctx->g.ctas == 2) ? 1 : 0;
        void* kern = frac ? (two ? (void*)k_sp_run<true, false, 2, true> : (void*)k_sp_run<true, false, 1, true>)
                          : (two ? (void*)k_sp_run<true, false, 2, false> : (void*)k_sp_run<true, false, 1, false>);
        const int smem = two ? SweepCfg<2>::kSmem : SweepCfg<1>::kSmem;
        const int threads = two ? SweepCfg<2>::kThreads : SweepCfg<1>::kThreads;
        // (set on every launch: a per-device "already set" table would be shared, unsynchronised, by the worker threads of the
        //  multi-GPU predict path; the call costs a microsecond)
        PDP_CUDA_CHECK(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, smem));
        if (two) PDP_CUDA_CHECK(cudaMemsetAsync(ctx->s.sm_ctr, 0, sizeof(int32_t) * PDP_MAX_SMS, stream));
        PDP_CUDA_CHECK(cudaLaunchCooperativeKernel(kern, dim3(ctx->num_sms * (two ? 2 : 1)), dim3(threads), args, smem, stream));
    } else {
        void* kern = prm.full_state ? (frac ? (void*)k_sp_run<false, true, 1, true> : (void*)k_sp_run<false, true, 1, false>)
                                    : (frac ? (void*)k_sp_run<false, false, 1, true> : (void*)k_sp_run<false, false, 1, false>);
        int blocks = coop_blocks(ctx, kern);
        if (blocks < 1) { pdp_set_error("pdp_sp_run: occupancy query failed"); return PDP_ERR_CUDA; }
        PDP_CUDA_CHECK(cudaLaunchCooperativeKernel(kern, dim3(blocks), dim3(256), args, 0, stream));
    }
    PDP_LAUNCH_CHECK(ctx);
    return PDP_OK;
}

extern "C" int pdp_simplify(pdp_ctx* ctx, void* stream_) {
    if (!ctx) { pdp_set_error("pdp_simplify: null context"); return PDP_ERR_ARG; }
    KArgs A = make_args(ctx);
    void* args[] = {&A};
    int blocks = coop_blocks(ctx, k_simplify);
    if (blocks < 1) { pdp_set_error("pdp_simplify: occupancy query failed"); return PDP_ERR_CUDA; }
    PDP_CUDA_CHECK(cudaLaunchCooperativeKernel((void*)k_simplify, dim3(blocks), dim3(256), args, 0, (cudaStream_t)stream_));
    PDP_LAUNCH_CHECK(ctx);
    return PDP_OK;
}

extern "C" int pdp_set_variables(pdp_ctx* ctx, const float* d_assignment, void* stream_) {
    if (!ctx || (!d_assignment && ctx->g.V > 0)) { pdp_set_error("pdp_set_variables: null argument"); return PDP_ERR_ARG; }
    KArgs A = make_args(ctx);
    void* args[] = {&A, &d_assignment};
    int blocks = coop_blocks(ctx, k_set_variables);
    if (blocks < 1) { pdp_set_error("pdp_set_variables: occupancy query failed"); return PDP_ERR_CUDA; }
    PDP_CUDA_CHECK(cudaLaunchCooperativeKernel((void*)k_set_variables, dim3(blocks), dim3(256), args, 0, (cudaStream_t)stream_));
    PDP_LAUNCH_CHECK(ctx);
    return PDP_OK;
}

static bool valid_fraction(float f) { return f == f && f >= 0.f && f < 1.f; }

// SP-inspired decimation (pdp_b200.h): the fraction of each problem's active variables the fused loop fixes per step
extern "C" int pdp_set_decimation_fraction(pdp_ctx* ctx, float fraction) {
    if (!ctx) { pdp_set_error("pdp_set_decimation_fraction: null context"); return PDP_ERR_ARG; }
    if (!valid_fraction(fraction)) { pdp_set_error("pdp_set_decimation_fraction: fraction %g not in [0, 1)", (double)fraction); return PDP_ERR_ARG; }
    ctx->dec_fraction = fraction;
    return PDP_OK;
}

extern "C" int pdp_decimation_select(pdp_ctx* ctx, const float* d_coeff, const float* d_score, const uint8_t* d_problem_sel,
                                     float fraction, float* d_assignment, void* stream_) {
    if (!ctx || (ctx->g.V > 0 && (!d_coeff || !d_score || !d_assignment))) { pdp_set_error("pdp_decimation_select: null argument"); return PDP_ERR_ARG; }
    if (!valid_fraction(fraction)) { pdp_set_error("pdp_decimation_select: fraction %g not in [0, 1)", (double)fraction); return PDP_ERR_ARG; }
    KArgs A = make_args(ctx);
    A.dec_fraction = fraction;
    void* args[] = {&A, &d_coeff, &d_score, &d_problem_sel, &d_assignment};
    int blocks = coop_blocks(ctx, k_decimation_select);
    if (blocks < 1) { pdp_set_error("pdp_decimation_select: occupancy query failed"); return PDP_ERR_CUDA; }
    PDP_CUDA_CHECK(cudaLaunchCooperativeKernel((void*)k_decimation_select, dim3(blocks), dim3(256), args, 0, (cudaStream_t)stream_));
    PDP_LAUNCH_CHECK(ctx);
    return PDP_OK;
}

// conflict rollback (pdp_b200.h)
extern "C" size_t pdp_rollback_scratch_bytes(int64_t V, int64_t F, int64_t B) {
    if (V < 0 || F < 0 || B < 0) return 0;
    return rb_layout(V, F, B).total;
}

extern "C" int pdp_set_conflict_rollback(pdp_ctx* ctx, void* d_scratch, size_t bytes) {
    if (!ctx) { pdp_set_error("pdp_set_conflict_rollback: null context"); return PDP_ERR_ARG; }
    if (d_scratch) {
        const size_t need = rb_layout(ctx->g.V, ctx->g.F, ctx->g.B).total;
        if (bytes < need) {
            pdp_set_error("pdp_set_conflict_rollback: scratch of %zu bytes, %zu needed", bytes, need);
            return PDP_ERR_WORKSPACE;
        }
        if ((uintptr_t)d_scratch % 16) { pdp_set_error("pdp_set_conflict_rollback: scratch not 16-byte aligned"); return PDP_ERR_ARG; }
    }
    ctx->rb_scratch = d_scratch;
    return PDP_OK;
}

extern "C" int pdp_get_rollbacks(pdp_ctx* ctx, int32_t* d_count, int32_t* d_last_iter, void* stream_) {
    if (!ctx) { pdp_set_error("pdp_get_rollbacks: null context"); return PDP_ERR_ARG; }
    cudaStream_t stream = (cudaStream_t)stream_;
    const size_t n = sizeof(int32_t) * (size_t)ctx->g.B;
    if (d_count && n) PDP_CUDA_CHECK(cudaMemcpyAsync(d_count, ctx->s.rb_count, n, cudaMemcpyDeviceToDevice, stream));
    if (d_last_iter && n) PDP_CUDA_CHECK(cudaMemcpyAsync(d_last_iter, ctx->s.rb_last, n, cudaMemcpyDeviceToDevice, stream));
    return PDP_OK;
}

extern "C" int pdp_debug_check_edge_mask(pdp_ctx* ctx, int32_t* d_errs, void* stream_) {
    if (!ctx || !d_errs) { pdp_set_error("pdp_debug_check_edge_mask: null argument"); return PDP_ERR_ARG; }
    cudaStream_t stream = (cudaStream_t)stream_;
    PDP_CUDA_CHECK(cudaMemsetAsync(d_errs, 0, 2 * sizeof(int32_t), stream));
    KArgs A = make_args(ctx);
    k_check_edge_mask<<<pdp_grid(ctx->g.V, 256, ctx->num_sms), 256, 0, stream>>>(A, d_errs);
    PDP_LAUNCH_CHECK(ctx);
    return PDP_OK;
}

extern "C" int pdp_trace_length(pdp_ctx* ctx, int32_t* host_out, void* stream_) {
    if (!ctx || !host_out) { pdp_set_error("pdp_trace_length: null argument"); return PDP_ERR_ARG; }
    cudaStream_t stream = (cudaStream_t)stream_;
    PDP_CUDA_CHECK(cudaMemcpyAsync(host_out, ctx->s.ctrl + CTRL_TRACE_LEN, sizeof(int32_t), cudaMemcpyDeviceToHost, stream));
    PDP_CUDA_CHECK(cudaStreamSynchronize(stream));
    return PDP_OK;
}
