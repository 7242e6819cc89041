// pdp_walksat.cu -- WalkSAT post-processing (reference pdp/nn/solver.py:433-467 + 388-399) as one
// persistent cooperative kernel.
//
// The reference recomputes, every iteration and for the whole batch, the clause energies (5 SpMM), the
// per-variable energy deltas (7 SpMM) and two dense [V,B] arg-max matrices -- to flip ONE variable per
// unsatisfied problem.  Here the per-clause literal sums, the per-variable break-minus-make deltas and
// the per-variable "sits in an unsatisfied clause" counts are built once and then maintained
// incrementally by the thread that flips a problem's variable (integers: exact, order independent), so an
// iteration costs one streaming selection pass over the variables (12 B per variable) plus O(degree * k)
// updates per problem.  Selection follows the reference exactly: greedy = first index of the minimum
// delta over ALL variables of the problem, random = first index of the maximum of fl(fl(x - min x) + 1)
// with x = [variable in an unsatisfied clause] * r, coin = r_b > epsilon.
#include <stdlib.h>

#include "pdp_device.cuh"


namespace {

// Philox-4x32-10 counter based generator: (seed, counter) -> uniform float in [0,1)
__device__ __forceinline__ float philox_uniform(uint64_t seed, uint32_t c0, uint32_t c1, uint32_t c2) {
    uint32_t k0 = (uint32_t)seed, k1 = (uint32_t)(seed >> 32);
    uint32_t x0 = c0, x1 = c1, x2 = c2, x3 = 0x5eed5eedu;
#pragma unroll
    for (int rnd = 0; rnd < 10; ++rnd) {
        const uint32_t hi0 = __umulhi(0xD2511F53u, x0), lo0 = 0xD2511F53u * x0;
        const uint32_t hi1 = __umulhi(0xCD9E8D57u, x2), lo1 = 0xCD9E8D57u * x2;
        const uint32_t y0 = hi1 ^ x1 ^ k0, y1 = lo1, y2 = hi0 ^ x3 ^ k1, y3 = lo0;
        x0 = y0; x1 = y1; x2 = y2; x3 = y3;
        k0 += 0x9E3779B9u; k1 += 0xBB67AE85u;
    }
    return (float)(x0 >> 8) * (1.0f / 16777216.0f);
}

struct WsArgs {
    int32_t W;
    float epsilon;
    int32_t rep;
    const float* rand_var;    // [W,V] or null
    const float* rand_coin;   // [W,B] or null
    uint64_t seed;
    float* prediction;        // [V]
    int32_t* iters_done;
    int32_t cta_loop;         // CTA-per-problem search loop (no replication, contiguous problems)
};

__device__ __forceinline__ float ws_rand_var(const WsArgs& w, int it, int64_t i, int64_t V) {
    return w.rand_var ? w.rand_var[(int64_t)it * V + i] : philox_uniform(w.seed, (uint32_t)i, (uint32_t)it, 0x76617231u);
}
__device__ __forceinline__ float ws_rand_coin(const WsArgs& w, int it, int64_t b, int64_t B) {
    return w.rand_coin ? w.rand_coin[(int64_t)it * B + b] : philox_uniform(w.seed, (uint32_t)b, (uint32_t)it, 0x636f696eu);
}

// per-variable state kept in the closure scratch arrays (idle outside unit propagation)
#define WS_DELTA(s) ((s).up_cnt)   // [V] energy delta of flipping the variable (break - make)
#define WS_UVC(s) ((s).up_ev)      // [V] unsatisfied clauses the variable occurs in, times active

// flips variable `ind` of problem b and repairs every quantity that depends on it
__device__ void ws_flip(const pdp_graph& g, const pdp_state& s, int b, int ind) {
    const int a_old = (int)s.asg[ind];
    if (a_old == 0) return;   // inactive variable: flipping 0 is a no-op (solver.py:465)
    const int vb = g.var_ptr[ind], ve = g.var_ptr[ind + 1];
    int d_energy = 0;
    for (int p = vb; p < ve; ++p) {
        const int c = g.v_cls[p];
        if (!s.af[c] || (s.single[c] & 2)) continue;   // inactive clause, or clause already handled (duplicate literal)
        const int cb = g.cl_ptr[c], ce = g.cl_ptr[c + 1];
        int lsum = 0;
        for (int e = cb; e < ce; ++e) {
            const uint32_t w = g.c_var[e];
            if ((int)(w & PDP_IDX_MASK) == ind) lsum += (w & PDP_SIGN_BIT) ? -a_old : a_old;
        }
        const int agg_old = s.ws_true[c], deg = s.ws_deg[c];
        const int agg_new = agg_old - 2 * lsum;
        const int u_old = s.single[c] & 1, u_new = (agg_new == -deg) ? 1 : 0;
        for (int e = cb; e < ce; ++e) {
            const uint32_t w = g.c_var[e];
            const int j = (int)(w & PDP_IDX_MASK);
            if (!s.av[j]) continue;
            const int aj = (int)s.asg[j];   // still the old value for j == ind
            const int lit_old = (w & PDP_SIGN_BIT) ? -aj : aj;
            const int lit_new = (j == ind) ? -lit_old : lit_old;
            const int c_old = (agg_old - lit_old == 1 - deg) ? lit_old : 0;
            const int c_new = (agg_new - lit_new == 1 - deg) ? lit_new : 0;
            if (c_new != c_old) WS_DELTA(s)[j] += c_new - c_old;
            if (u_new != u_old) WS_UVC(s)[j] += u_new - u_old;
        }
        s.ws_true[c] = agg_new;
        s.single[c] = (uint8_t)(u_new | 2);
        d_energy += u_new - u_old;
    }
    for (int p = vb; p < ve; ++p) s.single[g.v_cls[p]] &= 1;   // clear the visit marks
    s.asg[ind] = (int8_t)(-a_old);
    s.energy[b] += d_energy;
}

// ------------------------------------------------------------------------------------------------
// CTA-per-problem search loop (no batch replication, problems contiguous in the batch).  Problems never
// interact, so a CTA runs all W iterations of its problem without any grid-wide barrier.  Per iteration
// the reference needs, per problem, (a) the first index of the minimum energy delta over all variables
// and (b) a random variable that sits in an unsatisfied clause.  Both come from per-chunk summaries
// (min (delta, index) key and candidate count per chunk of the problem's variables) held in shared
// memory and repaired after every flip for the handful of chunks the flip touched, so an iteration costs
// O(n / chunk + chunk * touched) instead of a pass over all n variables.
//   injected draws (parity mode): (b) is the reference's arg-max of fl(fl(x - min x) + 1) over ALL
//   variables, x = [in an unsatisfied clause] * r_i -- an exact O(n) scan by the CTA;
//   counter-based generator: (b) is the k-th candidate, k uniform -- the same distribution.
// Mutable arrays are read with __ldcg: they are updated with L2 atomics by this same CTA.
// ------------------------------------------------------------------------------------------------
#define WS_NB 2048   // max chunks per problem
struct WsSmem {
    unsigned long long smin[WS_NB];
    int scount[WS_NB];
    uint32_t dirty[WS_NB / 32];
    unsigned long long r64[2][8];
    uint32_t r32[2][8];
    int energy, pick, total;
};

__device__ __forceinline__ unsigned long long ws_gkey(int delta, int64_t i) {
    return ((unsigned long long)(uint32_t)(delta + 0x40000000) << 32) | (uint32_t)i;
}

// summary of chunk `blk` of the problem [pv0, pv1): executed by one warp
__device__ __forceinline__ void ws_chunk_summary(const pdp_state& s, WsSmem& sm, int pv0, int pv1, int bs, int blk) {
    const int lo = pv0 + blk * bs, hi = min(lo + bs, pv1);
    unsigned long long key = ~0ull;
    int cnt = 0;
    for (int i = lo + lane_id(); i < hi; i += 32) {
        const int d = __ldcg(&WS_DELTA(s)[i]), u = __ldcg(&WS_UVC(s)[i]);
        const unsigned long long k = ws_gkey(d, i);
        key = k < key ? k : key;
        cnt += (u > 0) ? 1 : 0;
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) { const unsigned long long k2 = shfl_xor_u64(key, o); key = k2 < key ? k2 : key; }
    cnt = __reduce_add_sync(0xffffffffu, cnt);
    if (lane_id() == 0) { sm.smin[blk] = key; sm.scount[blk] = cnt; }
}

// flips variable `ind` (all threads of the CTA), repairing clause sums, deltas, counts, chunk dirty bits
__device__ __forceinline__ void ws_flip_cta(const pdp_graph& g, const pdp_state& s, WsSmem& sm, int pv0, int bs, int ind) {
    const int a_old = (int)__ldcg(&s.asg[ind]);
    if (a_old != 0) {   // flipping an inactive variable (0) is a no-op (solver.py:465)
        const int vb = g.var_ptr[ind], ve = g.var_ptr[ind + 1];
        for (int p = vb + (int)threadIdx.x; p < ve; p += (int)blockDim.x) {
            const int c = g.v_cls[p];
            if (!s.af[c]) continue;
            bool dup = false;   // the clause already handled through an earlier occurrence of the variable
            for (int p2 = vb; p2 < p; ++p2) dup |= (g.v_cls[p2] == c);
            if (dup) continue;
            const int cb = g.cl_ptr[c], ce = g.cl_ptr[c + 1];
            int lsum = 0;
            for (int e = cb; e < ce; ++e) {
                const uint32_t w = g.c_var[e];
                if ((int)(w & PDP_IDX_MASK) == ind) lsum += (w & PDP_SIGN_BIT) ? -a_old : a_old;
            }
            const int agg_old = __ldcg(&s.ws_true[c]), deg = s.ws_deg[c];
            const int agg_new = agg_old - 2 * lsum;
            const int u_old = __ldcg(&s.single[c]) & 1, u_new = (agg_new == -deg) ? 1 : 0;
            for (int e = cb; e < ce; ++e) {
                const uint32_t w = g.c_var[e];
                const int j = (int)(w & PDP_IDX_MASK);
                if (!s.av[j]) continue;
                const int aj = (int)__ldcg(&s.asg[j]);   // still the old value for j == ind
                const int lit_old = (w & PDP_SIGN_BIT) ? -aj : aj;
                const int lit_new = (j == ind) ? -lit_old : lit_old;
                const int c_old = (agg_old - lit_old == 1 - deg) ? lit_old : 0;
                const int c_new = (agg_new - lit_new == 1 - deg) ? lit_new : 0;
                if (c_new != c_old) atomicAdd(&WS_DELTA(s)[j], c_new - c_old);
                if (u_new != u_old) atomicAdd(&WS_UVC(s)[j], u_new - u_old);
                if (c_new != c_old || u_new != u_old) { const int k = (j - pv0) / bs; atomicOr(&sm.dirty[k >> 5], 1u << (k & 31)); }
            }
            __stcg(&s.ws_true[c], agg_new);
            __stcg(&s.single[c], (uint8_t)u_new);
            if (u_new != u_old) atomicAdd(&sm.energy, u_new - u_old);
        }
    }
    __syncthreads();
    if (threadIdx.x == 0 && a_old != 0) __stcg(&s.asg[ind], (int8_t)(-a_old));
    __syncthreads();
}

__device__ void ws_problem_loop(const KArgs& A, const WsArgs& wa, WsSmem& sm, int b) {
    const pdp_graph& g = A.g; const pdp_state& s = A.s;
    const int tid = threadIdx.x, nthr = blockDim.x, warp = tid >> 5, nwarp = nthr >> 5, lane = tid & 31;
    const int pv0 = g.prob_vptr[b], pv1 = g.prob_vptr[b + 1];
    const int n = pv1 - pv0;
    int it = 0;
    if (tid == 0) sm.energy = s.energy[b];
    __syncthreads();
    if (n > 0 && sm.energy > 0) {
        int bs = 32;
        while ((n + bs - 1) / bs > WS_NB) bs <<= 1;
        const int nblk = (n + bs - 1) / bs;
        for (int k = warp; k < nblk; k += nwarp) ws_chunk_summary(s, sm, pv0, pv1, bs, k);
        for (int k = tid; k < WS_NB / 32; k += nthr) sm.dirty[k] = 0u;
        __syncthreads();
        for (; it < wa.W && sm.energy > 0; ++it) {
            // ---- greedy candidate: first index of the minimum delta (solver.py:453-454)
            unsigned long long kg = ~0ull;
            int cnt = 0;
            for (int k = tid; k < nblk; k += nthr) { const unsigned long long v = sm.smin[k]; kg = v < kg ? v : kg; cnt += sm.scount[k]; }
#pragma unroll
            for (int o = 16; o > 0; o >>= 1) { const unsigned long long k2 = shfl_xor_u64(kg, o); kg = k2 < kg ? k2 : kg; }
            cnt = __reduce_add_sync(0xffffffffu, cnt);
            if (lane == 0) { sm.r64[0][warp] = kg; sm.r32[0][warp] = (uint32_t)cnt; }
            // ---- random candidate
            unsigned long long kr = 0ull;
            uint32_t mn = 0x7f800000u, mx = 0u;
            if (wa.rand_var) {
                for (int i = pv0 + tid; i < pv1; i += nthr) {
                    const float x = (__ldcg(&WS_UVC(s)[i]) > 0) ? wa.rand_var[(int64_t)it * g.V + i] : 0.f;
                    const unsigned long long k = ((unsigned long long)f2u(argmax_key(x, 0.f)) << 32) | (uint32_t)(0xffffffffu - (uint32_t)i);
                    kr = k > kr ? k : kr;
                    mn = min(mn, f2u(x)); mx = max(mx, f2u(x));
                }
#pragma unroll
                for (int o = 16; o > 0; o >>= 1) { const unsigned long long k2 = shfl_xor_u64(kr, o); kr = k2 > kr ? k2 : kr; }
                mn = __reduce_min_sync(0xffffffffu, mn); mx = __reduce_max_sync(0xffffffffu, mx);
                if (lane == 0) { sm.r64[1][warp] = kr; sm.r32[1][warp] = mn; sm.r32[0][warp] |= 0u; }
            }
            __syncthreads();
            for (int w2 = 0; w2 < nwarp; ++w2) { const unsigned long long v = sm.r64[0][w2]; kg = (w2 == 0 || v < kg) ? v : kg; }
            int total = 0;
            for (int w2 = 0; w2 < nwarp; ++w2) total += (int)sm.r32[0][w2];
            uint32_t ri;
            if (wa.rand_var) {
                for (int w2 = 0; w2 < nwarp; ++w2) { const unsigned long long v = sm.r64[1][w2]; kr = (w2 == 0 || v > kr) ? v : kr; mn = (w2 == 0) ? sm.r32[1][w2] : min(mn, sm.r32[1][w2]); }
                // max of x over the CTA (for the exact key when min x > 0)
                __syncthreads();
                if (lane == 0) sm.r32[1][warp] = mx;
                __syncthreads();
                for (int w2 = 0; w2 < nwarp; ++w2) mx = (w2 == 0) ? sm.r32[1][w2] : max(mx, sm.r32[1][w2]);
                ri = 0xffffffffu - (uint32_t)(kr & 0xffffffffull);
                if (mn != 0u && mn != 0x7f800000u) {
                    // min x > 0: the reference's key is fl(fl(x - min x) + 1): redo the pick exactly
                    const float m = u2f(mn);
                    const float kmax = argmax_key(u2f(mx), m);
                    uint32_t first = 0xffffffffu;
                    for (int i = pv0 + tid; i < pv1; i += nthr) {
                        const float x = (__ldcg(&WS_UVC(s)[i]) > 0) ? wa.rand_var[(int64_t)it * g.V + i] : 0.f;
                        if (argmax_key(x, m) == kmax) first = min(first, (uint32_t)i);
                    }
                    first = __reduce_min_sync(0xffffffffu, first);
                    __syncthreads();
                    if (lane == 0) sm.r32[1][warp] = first;
                    __syncthreads();
                    for (int w2 = 0; w2 < nwarp; ++w2) first = (w2 == 0) ? sm.r32[1][w2] : min(first, sm.r32[1][w2]);
                    ri = first;
                }
            } else {
                // k-th variable that sits in an unsatisfied clause, k uniform (no candidate: x is all zero
                // and the reference's arg-max returns the first variable of the problem)
                if (warp == 0) {
                    int pick = pv0;
                    if (total > 0) {
                        const float u = philox_uniform(wa.seed, (uint32_t)b, (uint32_t)it, 0x76617231u);
                        int k = (int)(u * (float)total);
                        if (k >= total) k = total - 1;
                        int blk = 0;   // chunk holding the k-th candidate: warp-wide running prefix
                        for (int base = 0; base < nblk; base += 32) {
                            const int c = (base + lane < nblk) ? sm.scount[base + lane] : 0;
                            int incl = c;
#pragma unroll
                            for (int o = 1; o < 32; o <<= 1) { const int t = __shfl_up_sync(0xffffffffu, incl, o); if (lane >= o) incl += t; }
                            const int tot32 = __shfl_sync(0xffffffffu, incl, 31);
                            if (k < tot32) {
                                const unsigned hit = __ballot_sync(0xffffffffu, k < incl);
                                const int l = __ffs(hit) - 1;
                                blk = base + l;
                                k -= __shfl_sync(0xffffffffu, incl - c, l);
                                break;
                            }
                            k -= tot32;
                        }
                        const int lo = pv0 + blk * bs, hi = min(lo + bs, pv1);
                        for (int base = lo; base < hi; base += 32) {
                            const int i = base + lane;
                            const bool cand = (i < hi) && (__ldcg(&WS_UVC(s)[i]) > 0);
                            const unsigned m = __ballot_sync(0xffffffffu, cand);
                            const int c = __popc(m);
                            if (k < c) {
                                unsigned mm = m;
                                for (int q = 0; q < k; ++q) mm &= mm - 1;
                                pick = base + __ffs(mm) - 1;
                                break;
                            }
                            k -= c;
                        }
                    }
                    if (lane == 0) sm.pick = pick;
                }
                __syncthreads();
                ri = (uint32_t)sm.pick;
            }
            const uint32_t gi = (uint32_t)(kg & 0xffffffffull);
            const bool coin = ws_rand_coin(wa, it, b, g.B) > wa.epsilon;   // solver.py:460-461
            const uint32_t ind = coin ? gi : ri;
            __syncthreads();
            ws_flip_cta(g, s, sm, pv0, bs, (int)ind);
            // ---- repair the summaries of the chunks the flip touched
            for (int k = warp; k < nblk; k += nwarp) {
                if ((sm.dirty[k >> 5] >> (k & 31)) & 1u) ws_chunk_summary(s, sm, pv0, pv1, bs, k);
            }
            __syncthreads();
            for (int k = tid; k < (nblk + 31) / 32; k += nthr) sm.dirty[k] = 0u;
            __syncthreads();
        }
    }
    __syncthreads();
    if (tid == 0) {
        s.energy[b] = sm.energy;
        if (it > 0) atomicMax(&s.ctrl[CTRL_WS_ITERS], it);
    }
    __syncthreads();
}

// grid-wide search loop: every iteration is one pass over all variables of the batch plus grid barriers.
// Kept for batch replication (the reference stops ALL replicas at the iteration in which every original
// problem has a solved replica, solver.py:446-449 -- a batch-global condition) and for batches whose
// problems are not contiguous.
__device__ int ws_grid_loop(const KArgs& A, const WsArgs& wa, cg::grid_group& grid) {
    const pdp_graph& g = A.g; const pdp_state& s = A.s;
    const int rep = wa.rep > 1 ? wa.rep : 1;
    const int64_t B0 = g.B / rep;
    int it = 0;
#ifdef PDP_PHASE_TIMING
#define WS_T(slot_) do { if (gtid() == 0 && A.trace) { const long long _n = clock64(); atomicAdd(&A.trace[slot_], (int)((_n - _wt) >> 4)); _wt = _n; } } while (0)
    long long _wt = clock64();
#else
#define WS_T(slot_) do {} while (0)
#endif
    for (; it < wa.W; ++it) {
        const int slot = it & 1;
        if (!s.ctrl[CTRL_WS_UNSAT + slot]) break;
        WS_T(0);
        // ---- candidate selection: one streaming pass over (delta, count, r)
        {
            KeyedReducer<PickAcc> red;
            // the per-problem "still unsatisfied" flag is cached per lane: thousands of warps re-reading the
            // same few energy words every step would serialise on one L2 slice
            int cb = -1; bool cb_on = false;
            const int64_t stride = gwarps() * 32;
            for (int64_t i0 = gwarp() * 32 + lane_id(); i0 < g.V; i0 += 4 * stride) {
                int bb[4], dl[4], uv[4];
#pragma unroll
                for (int u = 0; u < 4; ++u) {
                    const int64_t i = i0 + u * stride;
                    const bool in = i < g.V;
                    bb[u] = in ? g.bvm[i] : -1;
                    dl[u] = in ? WS_DELTA(s)[i] : 0;
                    uv[u] = in ? WS_UVC(s)[i] : 0;
                }
#pragma unroll
                for (int u = 0; u < 4; ++u) {
                    const int64_t i = i0 + u * stride;
                    const int b = bb[u];
                    if (b < 0) continue;
                    if (b != cb) { cb = b; cb_on = s.energy[b] > 0; }
                    if (!cb_on) continue;
                    red.touch(s, b);
                    const float x = (uv[u] > 0) ? (1.f * ws_rand_var(wa, it, i, g.V)) : 0.f;
                    const unsigned long long kg = ((unsigned long long)(uint32_t)(dl[u] + 0x40000000) << 32) | (uint32_t)i;
                    const unsigned long long kr = ((unsigned long long)f2u(argmax_key(x, 0.f)) << 32) | (uint32_t)(0xffffffffu - (uint32_t)i);
                    red.acc.add(kg, kr, f2u(x));
                }
            }
            WS_T(1);
            red.finish(s);
        }
        if (gtid() == 0) { s.ctrl[CTRL_WS_UNSAT + (slot ^ 1)] = 0; s.ctrl[CTRL_WS_REDO + (slot ^ 1)] = 0; }
        WS_T(2);
        grid.sync();
        WS_T(3);
        // min x > 0 (every variable of the problem sits in an unsatisfied clause and drew r > 0): the
        // reference's key is fl(fl(x - min x) + 1), redo the random pick exactly
        WARP_STRIDED(b, g.B) {
            if (b >= g.B) continue;
            if (s.energy[b] > 0 && s.ws_best[2 * b] != 0u && s.ws_best[2 * b] != 0x7f800000u) {
                s.ctrl[CTRL_WS_REDO + slot] = 1;
                s.ws_key[2 * b + 1] = ~0ull;   // becomes an atomicMin over the index
            }
        }
        grid.sync();
        WS_T(4);
        if (s.ctrl[CTRL_WS_REDO + slot]) {
            WARP_STRIDED(i, g.V) {
                if (i >= g.V) continue;
                const int b = g.bvm[i];
                if (!(s.energy[b] > 0) || s.ws_best[2 * b] == 0u || s.ws_best[2 * b] == 0x7f800000u) continue;
                const float m = u2f(s.ws_best[2 * b]);
                const float kmax = argmax_key(u2f(s.ws_best[2 * b + 1]), m);
                const float x = ((WS_UVC(s)[i] > 0) ? 1.f : 0.f) * ws_rand_var(wa, it, i, g.V);
                if (argmax_key(x, m) == kmax) atomicMin(&s.ws_key[2 * b + 1], (unsigned long long)(uint32_t)i);
            }
            grid.sync();
        }
        // ---- flip one variable per unsatisfied problem (solver.py:460-465) and repair the state
        WARP_STRIDED(j, B0) {
            if (j >= B0) continue;
            bool all_unsat = true;
            for (int r = 0; r < rep; ++r) {
                const int64_t b = (int64_t)r * B0 + j;
                if (s.energy[b] > 0) {
                    const bool redo = (s.ws_best[2 * b] != 0u && s.ws_best[2 * b] != 0x7f800000u);
                    const uint32_t gi = (uint32_t)(s.ws_key[2 * b] & 0xffffffffull);
                    const uint32_t lo = (uint32_t)(s.ws_key[2 * b + 1] & 0xffffffffull);
                    const uint32_t ri = redo ? lo : (0xffffffffu - lo);
                    const bool coin = ws_rand_coin(wa, it, b, g.B) > wa.epsilon;
                    const uint32_t ind = coin ? gi : ri;
                    if (ind < (uint32_t)g.V) ws_flip(g, s, (int)b, (int)ind);
                }
                if (!(s.energy[b] > 0)) all_unsat = false;
                s.ws_key[2 * b] = ~0ull; s.ws_key[2 * b + 1] = 0ull; s.ws_best[2 * b] = 0x7f800000u; s.ws_best[2 * b + 1] = 0u;
            }
            if (all_unsat) s.ctrl[CTRL_WS_UNSAT + (slot ^ 1)] = 1;
        }
        WS_T(5);
        grid.sync();
        WS_T(6);
    }
    return it;
}

__global__ void __launch_bounds__(256) k_walksat(const __grid_constant__ KArgs A, const __grid_constant__ WsArgs wa) {
    cg::grid_group grid = cg::this_grid();
    const pdp_graph& g = A.g; const pdp_state& s = A.s;
    const int rep = wa.rep > 1 ? wa.rep : 1;
    const int64_t B0 = g.B / rep;
    // ---- set-up: assignment (solver.py:436-437), clause sums + energy (486-496), deltas (469-484)
    WARP_STRIDED(i, g.V) {
        if (i < g.V) s.asg[i] = s.av[i] ? ((s.sol[i] > 0.5f) ? (int8_t)1 : (int8_t)-1) : (int8_t)0;
    }
    WARP_STRIDED(b, g.B) { if (b < g.B) s.energy[b] = 0; }
    if (gtid() == 0) { s.ctrl[CTRL_WS_UNSAT] = 0; s.ctrl[CTRL_WS_UNSAT + 1] = 0; s.ctrl[CTRL_WS_REDO] = 0; s.ctrl[CTRL_WS_REDO + 1] = 0; }
    grid.sync();
    if (wa.W > 0) {
        KeyedReducer<EnergyAcc> red;
        WARP_STRIDED(a, g.F) {
            if (a >= g.F) continue;
            int agg = 0, deg = 0;
            for (int c = g.cl_ptr[a]; c < g.cl_ptr[a + 1]; ++c) {
                const uint32_t w = g.c_var[c];
                const int v = (int)(w & PDP_IDX_MASK);
                const int lit = (int)s.asg[v];
                agg += (w & PDP_SIGN_BIT) ? -lit : lit;
                deg += (lit != 0) ? 1 : 0;      // asg is 0 exactly for the inactive variables: no second gather of av
            }
            const bool unsat = (agg == -deg) && s.af[a];
            s.ws_true[a] = agg; s.ws_deg[a] = deg; s.single[a] = unsat ? 1 : 0;
            if (unsat) { red.touch(s, g.bfm[a]); red.acc.n += 1; }
        }
        red.finish(s);
    }
    grid.sync();
    if (wa.W > 0) {
        WARP_STRIDED(i, g.V) {
            if (i >= g.V) continue;
            const int ai = (int)s.asg[i], avi = s.av[i];
            int delta = 0, uv = 0;
            for (int p = g.var_ptr[i]; p < g.var_ptr[i + 1]; ++p) {
                const int a = g.v_cls[p];
                const int lit = (g.v_cedge[p] & PDP_SIGN_BIT) ? -ai : ai;
                if (avi && s.af[a] && (s.ws_true[a] - lit == 1 - s.ws_deg[a])) delta += lit;
                uv += s.single[a];
            }
            WS_DELTA(s)[i] = delta; WS_UVC(s)[i] = uv * avi;
        }
        // which problems are still unsatisfied (solver.py:444-451); reset the selection keys
        WARP_STRIDED(j, B0) {
            if (j >= B0) continue;
            bool all_unsat = true;
            for (int r = 0; r < rep; ++r) if (!(s.energy[(int64_t)r * B0 + j] > 0)) all_unsat = false;
            if (all_unsat) s.ctrl[CTRL_WS_UNSAT] = 1;
            for (int r = 0; r < rep; ++r) {
                const int64_t b = (int64_t)r * B0 + j;
                s.ws_key[2 * b] = ~0ull; s.ws_key[2 * b + 1] = 0ull; s.ws_best[2 * b] = 0x7f800000u; s.ws_best[2 * b + 1] = 0u;
            }
        }
    }
    grid.sync();
    int it = 0;
    if (wa.cta_loop) {
        __shared__ WsSmem sm;
        if (gtid() == 0) s.ctrl[CTRL_WS_ITERS] = 0;
        grid.sync();
        if (wa.W > 0)
            for (int b = blockIdx.x; b < g.B; b += gridDim.x) ws_problem_loop(A, wa, sm, b);
        grid.sync();
        it = s.ctrl[CTRL_WS_ITERS];
    } else {
        it = ws_grid_loop(A, wa, grid);
    }
    // ---- solver.py:467 + _update_solution (solver.py:388-399)
    WARP_STRIDED(i, g.V) {
        if (i >= g.V) continue;
        const float avf = (float)s.av[i];
        const float walk = ((float)s.asg[i] + 1.f) / 2.0f;
        const float merged = avf * walk + (1.0f - avf) * s.sol[i];
        if (s.av[i]) { s.sol[i] = merged; s.ctrl[CTRL_NATIVE] = 0; }
        if (wa.prediction) wa.prediction[i] = merged;
        WS_DELTA(s)[i] = 0; WS_UVC(s)[i] = 0;
    }
    WARP_STRIDED(a, g.F) { if (a < g.F) s.single[a] = 0; }
    WARP_STRIDED(b, g.B) { if (b < g.B) { s.energy[b] = 0; s.dirty[b] = 1; } }
    if (gtid() == 0) {
        s.ctrl[CTRL_WS_ITERS] = it; s.ctrl[CTRL_ANY_DIRTY] = 1;
        if (wa.iters_done) *wa.iters_done = it;
    }
}

}  // namespace

extern "C" int pdp_walksat(pdp_ctx* ctx, int32_t W, float epsilon, int32_t batch_replication, const float* d_rand_var,
                           const float* d_rand_coin, uint64_t seed, float* d_prediction, int32_t* d_iters_done, void* stream_) {
    if (!ctx) { pdp_set_error("pdp_walksat: null context"); return PDP_ERR_ARG; }
    if (W < 0) { pdp_set_error("pdp_walksat: negative iteration count"); return PDP_ERR_ARG; }
    if ((d_rand_var == nullptr) != (d_rand_coin == nullptr)) { pdp_set_error("pdp_walksat: rand_var and rand_coin must both be given or both be null"); return PDP_ERR_ARG; }
    const int rep = batch_replication > 1 ? batch_replication : 1;
    if (ctx->g.B % rep != 0) { pdp_set_error("pdp_walksat: batch size not divisible by replication"); return PDP_ERR_ARG; }
    KArgs A;
    A.g = ctx->g; A.s = ctx->s; A.trace = nullptr; A.trace_cap = 0; A.stagger_c = 0; A.stagger_v = 0; A.dec_fraction = 0.f;
#ifdef PDP_PHASE_TIMING
    A.trace = ctx->trace;
#endif
    WsArgs wa;
    wa.W = W; wa.epsilon = epsilon; wa.rep = rep; wa.rand_var = d_rand_var; wa.rand_coin = d_rand_coin; wa.seed = seed;
    wa.prediction = d_prediction; wa.iters_done = d_iters_done;
    // injected draws make the random pick an exact O(n) scan per iteration: one CTA per problem only while
    // problems are small; large problems with injected draws keep the grid-wide pass
    const bool small_or_generated = (d_rand_var == nullptr) || (ctx->g.B > 0 && ctx->g.V / ctx->g.B <= 32768);
    wa.cta_loop = (rep == 1 && ctx->g.prob_vptr != nullptr && ctx->g.contiguous_problems && small_or_generated &&
                   getenv("PDP_B200_WS_GRID") == nullptr) ? 1 : 0;
    void* args[] = {&A, &wa};
    int per_sm = 0;
    if (cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, k_walksat, 256, 0) != cudaSuccess || per_sm < 1) {
        pdp_set_error("pdp_walksat: occupancy query failed"); return PDP_ERR_CUDA;
    }
    if (per_sm > 4) per_sm = 4;
    PDP_CUDA_CHECK(cudaLaunchCooperativeKernel((void*)k_walksat, dim3(per_sm * ctx->num_sms), dim3(256), args, 0, (cudaStream_t)stream_));
    PDP_LAUNCH_CHECK(ctx);
    return PDP_OK;
}
