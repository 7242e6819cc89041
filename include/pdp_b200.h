/*
 * pdp_b200.h -- C ABI of libpdp_b200.so: the B200 (sm_100a) implementation of SATYR's factor-graph
 * message-passing hot path (microsoft/PDP-Solver).  Plain pointers and sizes only; no torch types.
 *
 * The reference has no FFI of its own: the boundary it exposes is the Python operator interface of
 * `pdp.nn.solver`, `pdp.nn.pdp_propagate`, `pdp.nn.pdp_decimate`, `pdp.nn.pdp_predict` and
 * `pdp.nn.util` (SURVEY.md section 8b).  Every entry point below names the reference operator
 * (file:line under /root/reference/src) whose arithmetic it replaces; the ctypes binding a
 * maintainer would add on the reference side is in INTEGRATION.md.
 *
 * Conventions
 *  - every pointer marked `d_` is a DEVICE pointer on the current CUDA device;
 *  - every call is asynchronous on `stream` (a cudaStream_t passed as void*) unless it says "syncs";
 *  - return value: 0 = ok, negative = error (pdp_last_error() gives the thread-local message);
 *  - no device allocation happens inside any call: the caller hands a workspace to pdp_create();
 *  - a context is bound to one device and must not be used from two threads at once.
 *
 * Tensor layouts at the boundary are the reference's batch tensors
 * (reference pdp/factorgraph/dataset.py:138-187):
 *    graph_map     int32 [2,E]  row 0 variable index, row 1 clause ("function") index, batch-global
 *    edge_feature  fp32  [E]    literal sign +1/-1
 *    batch_variable_map int32 [V], batch_function_map int32 [F]  problem id of each node
 * Message states are the reference's (variable_state [E,3], function_state [E,2]) pairs in the
 * caller's edge order.
 */
#ifndef PDP_B200_H
#define PDP_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef struct pdp_ctx pdp_ctx;

/* error codes */
#define PDP_OK 0
#define PDP_ERR_ARG (-1)
#define PDP_ERR_CUDA (-2)
#define PDP_ERR_WORKSPACE (-3)
#define PDP_ERR_UNSUPPORTED (-4)

/* per-problem flag bits reported by pdp_get_problem_flags() */
#define PDP_FLAG_TRIVIAL 1u        /* surveys became trivial (pdp_decimate.py:127-133)            */
#define PDP_FLAG_SOLVED 2u         /* a satisfying assignment was found (trainer.py:150-162)      */
#define PDP_FLAG_CONTRADICTION 4u  /* NaN surveys: SP contradiction (pdp_propagate.py:215-216)    */
#define PDP_FLAG_UP_CONFLICT 8u    /* unit propagation conflict (solver.py:247-261)               */
#define PDP_FLAG_ROLLED_BACK 16u   /* a decimation step was undone (pdp_set_conflict_rollback)    */

const char* pdp_version(void);
const char* pdp_last_error(void);

/* ---- context: graph ingest, replaces SATProblem.setup_problem + _compute_* ------------------
 * reference pdp/nn/solver.py:28-54,101-178 (the 14 sparse COO incidence matrices become one
 * CSR (by clause) + one CSC (by variable) with stable, ascending-edge-index adjacency).          */
size_t pdp_workspace_bytes(int64_t E, int64_t V, int64_t F, int64_t B);
int pdp_create(pdp_ctx** out, const int32_t* d_graph_map, const float* d_edge_feature,
               const int32_t* d_batch_variable_map, const int32_t* d_batch_function_map,
               int64_t E, int64_t V, int64_t F, int64_t B,
               void* d_workspace, size_t workspace_bytes, void* stream);
int pdp_destroy(pdp_ctx* ctx);
/* resets SATProblem state (active masks = 1, solution = 0.5, solver.py:49-54) and the
 * SequentialDecimator module state (pdp_decimate.py:179-183) */
int pdp_reset(pdp_ctx* ctx, void* stream);

/* ---- stateless operators (caller's edge order, fp32 tensors like the reference's) ------------ */

/* SatCNFEvaluator.forward, reference pdp/nn/util.py:210-236.  d_pred [V] -> d_solved [B], d_n_unsat [B] */
int pdp_cnf_eval(pdp_ctx* ctx, const float* d_pred, float* d_solved, float* d_n_unsat, void* stream);

/* the same without a context, straight on the caller's edge list (any edge order): the form `SatCNFEvaluator` is called in
 * by `_post_process_predictions` (reference pdp/trainer.py:125-148) on batches no solver context exists for.
 * d_graph_map int32 [2,E], d_edge_feature [E], d_bfm [F]; d_scratch: pdp_cnf_eval_edges_scratch_bytes(F, B) bytes. */
size_t pdp_cnf_eval_edges_scratch_bytes(int64_t F, int64_t B);
int pdp_cnf_eval_edges(const int32_t* d_graph_map, const float* d_edge_feature, const int32_t* d_batch_function_map,
                       int64_t E, int64_t V, int64_t F, int64_t B, const float* d_pred,
                       float* d_solved, float* d_n_unsat, void* d_scratch, void* stream);

/* _compute_energy, reference pdp/nn/solver.py:486-496.  d_assignment [V] in {-1,0,1}, d_av [V],
 * d_af [F] float 0/1 -> d_energy [B], d_unsat_fn [F] */
int pdp_energy(pdp_ctx* ctx, const float* d_assignment, const float* d_av, const float* d_af,
               float* d_energy, float* d_unsat_fn, void* stream);

/* _compute_energy_diff, reference pdp/nn/solver.py:469-484.  d_edge_mask [E] -> d_delta [V] */
int pdp_energy_diff(pdp_ctx* ctx, const float* d_assignment, const float* d_av, const float* d_edge_mask,
                    float* d_delta, void* stream);

/* SurveyPropagator.forward (adaptors off), reference pdp/nn/pdp_propagate.py:139-221.
 * dec_*: decimator state (inputs); prop_*: propagator state (read for frozen problems only);
 * d_edge_mask: NULL or [E]; d_active: NULL or uint8 [B]; out_q3 [E,3], out_fs2 [E,2]. */
int pdp_sp_step(pdp_ctx* ctx, const float* d_dec_q3, const float* d_dec_fs2, const float* d_edge_mask,
                const float* d_prop_q3, const float* d_prop_fs2, const uint8_t* d_active, float pi,
                float* d_out_q3, float* d_out_fs2, void* stream);

/* SurveyPropagator.forward with the neural adaptors applied by the caller (model type p-nd-np), reference
 * pdp/nn/pdp_propagate.py:139-221 with include_adaptors=True: d_x_log [E] = logsigmoid(function_input_projector(.)),
 * d_eta_in [E] = sigmoid(variable_input_projector(.)[:,0]), d_ext_in [E] = sign(variable_input_projector(.)[:,1]);
 * the message arithmetic (edge mask, leave-one-out sums, frozen-problem blend) is the same as pdp_sp_step. */
int pdp_sp_step_adapted(pdp_ctx* ctx, const float* d_x_log, const float* d_eta_in, const float* d_ext_in,
                        const float* d_edge_mask, const float* d_prop_q3, const float* d_prop_fs2,
                        const uint8_t* d_active, float pi, float* d_out_q3, float* d_out_fs2, void* stream);

/* the segmented sums of MessageAggregator.forward, reference pdp/nn/util.py:51-77: d_state [E,channels] ->
 * d_node_sum [V or F, channels] = torch.mm(mask, state) (ascending edge order inside a node); d_edge_loo (nullable)
 * [E,channels] = torch.mm(mask_transpose, node_sum) - state (leave one out).  by_variable: 1 = variable_mask, 0 = function_mask */
int pdp_edge_aggregate(pdp_ctx* ctx, int32_t by_variable, const float* d_state, int32_t channels, float* d_node_sum,
                       float* d_edge_loo, void* stream);

/* Dense per-edge layers of the neural model types on the tensor cores (tcgen05.mma kind::tf32, three-term split = fp32
 * accuracy; csrc/pdp_edge_nn.cu).  Context-free.  The rows' input is the concatenation [x1 | x2 | x3] of up to three
 * row-major device arrays (k_i columns each, 0 = unused).  w_img / bias: the weights pre-split and pre-tiled and the padded
 * bias, built once per layer by pdp_solver_b200/nn/tensor_ops.py (n_blk * n_mma accumulator columns per pass -- a multiple of
 * 16, at most 256 for the dense layer and 320 for the GRU cell -- and `passes` passes over K).
 * pdp_edge_mlp_forward: out[rows, n_out] = act([x1|x2|x3] W^T + b) * row_mask -- the nn.Linear (+ F.logsigmoid, act = 1) calls
 *   of MessageAggregator.forward, reference pdp/nn/util.py:51-77, and of the classifiers (act = 0).
 * pdp_edge_gru_forward: out[rows, hidden] = torch.nn.GRUCell([x1|x2], h), blended with h where row_mask is 0 -- the two cells of
 *   NeuralDecimator.forward, reference pdp/nn/pdp_decimate.py:51-87.  A pass holds n_blk * n_mma / 4 hidden units, four
 *   accumulator columns each (r, z, W_in x, W_hn h of the unit side by side; bias in the same order).  out must not alias h.
 * Alignment: d_x1, d_x2, d_x3, d_h, d_out and d_row_mask need only be 4-byte (float) aligned; rows and arrays that are 8- or
 * 16-byte aligned take wider accesses, the others element-by-element ones.  d_w_img must be 16-byte aligned (PDP_ERR_ARG). */
int pdp_edge_nn_swizzle(void);   /* 1: the weight images use the 64-byte swizzled operand layout (nn/tensor_ops.py follows) */
int pdp_edge_nn_chunk_k(void);   /* K elements per chunk of the weight images (16): the host side tiles W accordingly */
int pdp_edge_mlp_forward(const float* d_x1, int32_t k1, const float* d_x2, int32_t k2, const float* d_x3, int32_t k3, int64_t rows,
                         const float* d_w_img, const float* d_bias, int32_t n_blk, int32_t n_mma, int32_t passes, int32_t n_out,
                         int32_t act, const float* d_row_mask, float* d_out, void* stream);
int pdp_edge_gru_forward(const float* d_x1, int32_t k1, const float* d_x2, int32_t k2, const float* d_h, int32_t hidden, int64_t rows,
                         const float* d_w_img, const float* d_bias, int32_t n_blk, int32_t n_mma, int32_t passes,
                         const float* d_row_mask, float* d_out, void* stream);

/* SurveyScorer.forward (adaptors off), reference pdp/nn/pdp_predict.py:155-192.
 * d_fs2 [E,2], d_af [F] -> d_score [V] */
int pdp_score(pdp_ctx* ctx, const float* d_fs2, const float* d_af, float pi, float* d_score, void* stream);

/* ---- solver state held by the context ------------------------------------------------------- */

/* loads (propagator_state, decimator_state) as get_init_state() returns them
 * (reference pdp/nn/solver.py:498-511) into the internal variable-major message arrays */
int pdp_load_state(pdp_ctx* ctx, const float* d_prop_q3, const float* d_prop_fs2,
                   const float* d_dec_q3, const float* d_dec_fs2, void* stream);
/* the same for a state whose every edge carries the same values, as get_init_state(randomized=False)
 * returns (reference pdp/nn/pdp_predict.py:203-206: variable_state = 1/3, function_state = [0.5, 0]) */
int pdp_load_state_const(pdp_ctx* ctx, float qu, float qs, float qd, float eta, float ext, void* stream);
/* writes the current message state in the caller's edge order: out_q3 [E,3], out_fs2 [E,2] 
 * Columns 1:3 of the [E,3] state (q_s, q_*) are tracked exactly only by a pdp_sp_run with full_state = 1; otherwise they are
 * re-derived on export from the previous surveys with the CURRENT masks: for a problem whose last iteration fixed a variable they
 * can differ from the reference's on the edges next to the fix (column 0, q_u, and the surveys are always exact; the predict path
 * reads neither). */
int pdp_store_state(pdp_ctx* ctx, float* d_out_q3, float* d_out_fs2, void* stream);
/* overwrite / read the SATProblem masks (float 0/1 like the reference's tensors); NULL = skip.  Node masks installed this
 * way count as the decimator's edge mask from the next sweep on (reference pdp/nn/solver.py:370-374). */
int pdp_set_masks(pdp_ctx* ctx, const float* d_av, const float* d_af, const float* d_solution, void* stream);
int pdp_get_masks(pdp_ctx* ctx, float* d_av, float* d_af, float* d_solution, float* d_is_sat,
                  uint8_t* d_active, float* d_edge_mask, void* stream);
/* installs the per-problem active mask (uint8 [B]) a caller's own termination callback produced between two
 * one-iteration pdp_sp_run calls (reference pdp/nn/solver.py:376-384) */
int pdp_set_active(pdp_ctx* ctx, const uint8_t* d_active, void* stream);
int pdp_get_problem_flags(pdp_ctx* ctx, uint32_t* d_flags, int32_t* d_counters, int32_t* d_freeze_iter, void* stream);

/* SATProblem.simplify / set_variables, reference pdp/nn/solver.py:180-285 (unit propagation and
 * pure-literal peeling to closure, on device, no host round trips). d_assignment [V] in {-1,0,1}. */
int pdp_simplify(pdp_ctx* ctx, void* stream);
int pdp_set_variables(pdp_ctx* ctx, const float* d_assignment, void* stream);

typedef struct {
    int32_t iterations;         /* T: iteration_num of forward()                        */
    float tolerance;            /* SequentialDecimator tolerance (config: 0.02)         */
    int32_t t_max;              /* SequentialDecimator t_max (config: 100)              */
    float pi;                   /* SP external-force strength (0 for p-d-p)             */
    int32_t check_termination;  /* 1 = trainer._check_recurrence_termination semantics  */
    int32_t batch_replication;  /* b of `-b`; problem id of replica r of j is r*B/b + j */
    int32_t full_state;         /* 1 = also keep q_s and q_* (the [E,3] state) exact    */
    int32_t flags;              /* bit 0: use the generic (thread per node) passes, not the blocked ones;
                                   bit 1: grid-wide decimation phases only (no CTA-local decimation);
                                   bit 2: full-scan UP / peel closure in those phases (not the frontier lists);
                                   bit 3: check_termination = 1 keeps the active mask (trivial-survey test, early exit)
                                          but leaves the solved-problem check to the caller (pdp_set_active) */
} pdp_sp_params;

/* PropagatorDecimatorSolverBase._forward_core for the p-d-p model, reference
 * pdp/nn/solver.py:355-386 = T x [ SurveyPropagator.forward ; SequentialDecimator.forward
 * (pdp_decimate.py:122-177, incl. SurveyScorer, set_variables and simplify) ; edge mask ;
 * IdentityPredictor + _update_solution ; _check_recurrence_termination (trainer.py:150-162) ]
 * in ONE persistent cooperative kernel with per-problem convergence/termination flags.
 * d_iters_done: device int32[1] receiving the number of iterations executed (NULL = skip).
 * Can be called repeatedly; module state (previous surveys, counters) persists until pdp_reset. */
int pdp_sp_run(pdp_ctx* ctx, const pdp_sp_params* params, int32_t* d_iters_done, void* stream);

/* SP-inspired decimation (Braunstein, Mezard, Zecchina, Random Structures & Algorithms 27, 2005), generalising the rule of
 * SequentialDecimator (reference pdp/nn/pdp_decimate.py:152-171, one arg-max variable per problem and step).  With a
 * fraction f in [0, 1), a problem b selected at a step (converged, active, no NaN coefficient, sum of coefficients > 0)
 * with A_b active variables takes K_b = max(1, floor((double)f * A_b)) variables:
 *   K_b == 1: the reference's arg-max rule (first index attaining the max of fl(fl(c - min) + 1));
 *   K_b >= 2: the first min(K_b, #candidates) of the active variables with c > 0, ordered by c descending, then index
 *             ascending (exact fp32 comparisons); each gets sign(score).
 * All variables of a step are fixed together (_set_variable_core, solver.py:205-226), then unit propagation and peeling run.
 * pdp_set_decimation_fraction: the fraction pdp_sp_run uses; 0 after pdp_create (the reference's rule), kept by pdp_reset;
 *   PDP_ERR_ARG unless 0 <= f < 1.
 * pdp_decimation_select: the same rule, stateless, on caller-supplied coefficients d_coeff [V] (>= 0; |score| * active *
 *   converged in the reference) and scores d_score [V]; d_problem_sel uint8 [B] (NULL = every problem) stands for
 *   "converged and active"; A_b counts the context's active variables.  d_assignment [V] receives sign(score) on the taken
 *   variables and 0 elsewhere.  Uses the context's per-step scratch: not concurrently with pdp_sp_run on the context. */
int pdp_set_decimation_fraction(pdp_ctx* ctx, float fraction);
int pdp_decimation_select(pdp_ctx* ctx, const float* d_coeff, const float* d_score, const uint8_t* d_problem_sel,
                          float fraction, float* d_assignment, void* stream);

/* Conflict rollback for SP-inspired decimation.  One unit-propagation conflict ends a problem (the `== 1` quirk of
 * solver.py:257,261 wipes it, any count sets PDP_FLAG_UP_CONFLICT), so a step that fixes too many variables at once throws
 * away every step before it.  With rollback on, each problem b carries a halving exponent h_b and a rollback count r_b
 * (both 0 after pdp_reset) and pdp_sp_run decimates with
 *   K_b = max(1, floor((double)f * A_b) >> h_b)      (h_b = 0: the rule of pdp_set_decimation_fraction; same selection).
 * When a step of b with K_b >= 2 fixes its variables and the UP + peel closure that follows sets PDP_FLAG_UP_CONFLICT,
 * which was clear before the step, b's active variables, active clauses, solution and is_sat go back to their values just
 * before the fix (the edge mask with them), the conflict bit is cleared, PDP_FLAG_ROLLED_BACK is set, and h_b and r_b grow
 * by one.  Messages, previous surveys and counters are untouched: the step changed none of them.  A K_b = 1 step that
 * conflicts stands (retrying it would pick the same variable from the same surveys).  h_b never decreases before
 * pdp_reset.  The decimation trace keeps the fixes of a rolled-back step.
 * pdp_rollback_scratch_bytes: bytes of the snapshot buffer (the state of the problems a step decimates, taken before the fix).
 * pdp_set_conflict_rollback: d_scratch (device, 16-byte aligned, >= pdp_rollback_scratch_bytes) turns rollback on, NULL
 *   turns it off; off after pdp_create, kept by pdp_reset.  The buffer belongs to the caller and must outlive its use.
 *   Rollback acts only when a decimation fraction is set.
 * pdp_get_rollbacks: d_count int32 [B] receives r_b, d_last_iter int32 [B] the iteration (1-based, counted since
 *   pdp_reset) of b's last rollback, 0 when none; NULL = skip. */
size_t pdp_rollback_scratch_bytes(int64_t V, int64_t F, int64_t B);
int pdp_set_conflict_rollback(pdp_ctx* ctx, void* d_scratch, size_t bytes);
int pdp_get_rollbacks(pdp_ctx* ctx, int32_t* d_count, int32_t* d_last_iter, void* stream);

/* Model type `reinforce` (SP with the reinforcement term, Chavas, Furtlehner, Mezard, Zecchina, J. Stat. Mech. 2005;
 * reference ReinforceSurveyPropagatorSolver, solver.py:598-610) in pdp_sp_run.  With the mode on, iteration k of the runs
 * since pdp_set_reinforce (k = 0, 1, ...) is, in the reference's order (solver.py:355-386):
 *   1. the SP sweep with params->pi and the external forces ext = function_state[:,1] as input (as without the mode);
 *   2. with check_termination, previous surveys and at least one active variable in the batch: a still-active problem whose
 *      sparse_max(smooth-max_i(|eta_prev - eta| * em) * av) (per-problem min, the p-d-p convergence statistic) is <= 0.01
 *      retires (ReinforceDecimator, pdp_decimate.py:204-215); its freeze iteration is recorded;
 *   3. if d_coins[k] < decimation_probability: every variable is scored (SurveyScorer with pi, pdp_score) from the new
 *      surveys and the current forces, and every edge of variable i takes ext = sign(score_i): on all edges without
 *      check_termination, else as m * sign + (1 - m) * ext with m = 1 iff the problem is active after step 2;
 *   4. with check_termination: an active variable's solution becomes [sum of its forces > 0] (ReinforcePredictor +
 *      _update_solution) -- on the run's first iteration and where step 3 ran, the only iterations it can change;
 *   5. with check_termination and flags bit 3 clear: the termination check of the p-d-p loop (trainer.py:150-162, a solved
 *      replica retires its problem) on the problems step 4 touched.
 * No variable is fixed; tolerance, t_max, the decimation fraction and conflict rollback are not used.  Without full_state
 * the run takes the blocked passes where the batch allows them, with the pi terms per variable: this needs the forces
 * loaded by pdp_load_state to be the same on all edges of each variable (step 3 keeps them so); when they are not, the
 * runs take the generic passes until the next load.  Without full_state, pdp_store_state re-derives q_s and q_* with the
 * forces the last sweep read (before that iteration's coin).  d_coins: device fp32, n_coins of them, owned by the caller
 * until the mode is turned off; NULL turns the mode off.  Off after pdp_create; pdp_reset keeps the mode and the coin
 * index k.  pdp_sp_run returns PDP_ERR_ARG when the iterations of the runs since pdp_set_reinforce, each run counted with
 * all of its params->iterations, would exceed n_coins. */
int pdp_set_reinforce(pdp_ctx* ctx, const float* d_coins, int32_t n_coins, float decimation_probability);

/* IdentityPredictor.forward(last_call=True), reference pdp/nn/pdp_predict.py:118-128.
 * pdp_count_active_variables syncs the stream.  d_draws holds >= n_active uniform draws that are
 * consumed by the active variables in batch-global variable order (like torch.rand(n_active)). */
int pdp_count_active_variables(pdp_ctx* ctx, int64_t* host_out, void* stream);
int pdp_random_fill(pdp_ctx* ctx, const float* d_draws, void* stream);

/* _local_search (WalkSAT) + _update_solution, reference pdp/nn/solver.py:433-467,388-399.
 * d_rand_var [W,V] / d_rand_coin [W,B]: the torch.rand draws of each iteration in the reference's
 * order; when both are NULL a counter-based generator seeded by `seed` is used instead.
 * d_prediction [V] receives the merged prediction; d_iters_done int32[1] (nullable). */
int pdp_walksat(pdp_ctx* ctx, int32_t W, float epsilon, int32_t batch_replication,
                const float* d_rand_var, const float* d_rand_coin, uint64_t seed,
                float* d_prediction, int32_t* d_iters_done, void* stream);

/* _deduplicate, reference pdp/nn/solver.py:401-431: d_prediction [V] (b replicas) ->
 * d_out_prediction [V/b], d_winner int32 [B/b] (replica index with minimum energy, first on ties) */
int pdp_deduplicate(pdp_ctx* ctx, int32_t batch_replication, const float* d_prediction,
                    float* d_out_prediction, int32_t* d_winner, void* stream);

/* optional recording of decimation events (tests): triples (iteration, variable, sign) appended to
 * d_trace, at most capacity_events of them; the running count is returned by pdp_trace_length (syncs) */
int pdp_set_trace_buffer(pdp_ctx* ctx, int32_t* d_trace, int32_t capacity_events);
int pdp_trace_length(pdp_ctx* ctx, int32_t* host_out, void* stream);

/* self-check of the blocked message layout built by pdp_create (tests): d_errs device int32[8] receives
 * the number of violated invariants per class (pdp_layout.cu; [6] and [7] must equal E when the
 * blocked layout is on); host_info int32[5] (nullable) = {blocked, variable blocks, clause blocks,
 * variable block stride, clause block stride} */
int pdp_debug_check_layout(pdp_ctx* ctx, int32_t* d_errs, int32_t* host_info, void* stream);
/* self-check of the edge-mask bits the sweeps read (tests): d_errs device int32[2] receives the number of edges whose bit in
 * the variable-side / clause-side layout differs from "variable or clause inactive" under the current node masks */
int pdp_debug_check_edge_mask(pdp_ctx* ctx, int32_t* d_errs, void* stream);

/* ---- host-side ingest helpers (no device work; SURVEY.md section 8f rank 1) ---------------------------
 * pdp_host_parse_ints: scans `text[0..len)` for decimal integers (optional leading '-', any other byte is a
 * separator) and writes the first `cap` of them to `out`; returns how many the text holds (so a caller may
 * size with cap = 0 first), -1 on bad arguments, -2 on a value beyond int32.  Replaces json.loads +
 * np.array(list) of one compact-JSON row (src/pdp/factorgraph/dataset.py:120-136).
 * pdp_host_parse_dimacs: streaming DIMACS CNF scanner (replaces the dense [m,n] clause matrix of
 * src/dimacs2json.py:24-50): literals are written to `lits` with their 0 terminators kept; `c` lines and the
 * `p cnf` line are skipped, `%` ends the file; info[0..3] = declared variables, declared clauses (-1 if no
 * header), entries written, clauses seen.  PDP_ERR_WORKSPACE if `cap` entries are not enough (info[2] = need). */
int64_t pdp_host_parse_ints(const char* text, int64_t len, int32_t* out, int64_t cap);
/* pdp_host_parse_rows: a whole compact-JSON file (one `[[n, m], [literals], [clauses], label, [id]]` row per line,
 * src/pdp/factorgraph/dataset.py:120-136) in one pass: the two integer lists of every row back to back in lits / cls
 * (row r = [row_ptr[r], row_ptr[r+1])), nm[2r..] = n, m, label[r], tail[2r..] = byte range of the id list for the caller to
 * decode.  Returns the row count, -(line number) of the first malformed row, or -2^62 when a capacity is too small. */
int64_t pdp_host_parse_rows(const char* text, int64_t len, int32_t* lits, int32_t* cls, int64_t int_cap,
                            int64_t* row_ptr, int32_t* nm, double* label, int64_t* tail, int64_t row_cap);
int pdp_host_parse_dimacs(const char* text, int64_t len, int32_t* lits, int64_t cap, int64_t* info);

/* counters for bench.py: number of kernels this library launched on behalf of the context */
int64_t pdp_launch_count(pdp_ctx* ctx);

#ifdef __cplusplus
}
#endif
#endif /* PDP_B200_H */
