// pdp_device.cuh -- grid-wide phases of the p-d-p loop, shared by the persistent cooperative kernel
// (pdp_loop.cu) and by the step-wise entry points.  Every phase is a __device__ function executed
// by ALL threads of a cooperative grid; the caller separates phases with grid.sync().
//
// The SP sweep exists twice:
//  * blocked passes (blk_clause_pass / blk_var_pass): the product path.  One CTA per block of whole
//    nodes, messages staged through shared memory, contiguous global reads and piece-wise contiguous
//    global writes (layout: pdp_common.cuh, DESIGN.md);
//  * generic passes (gen_*): thread per node with per-edge indexed global accesses into the same
//    layout.  They serve what the blocked passes leave out: the full [E,3] state, pi != 0, graphs whose
//    node degrees do not fit a block, and the problems on the sticky-NaN path.
//
// Work distribution of everything else: "warp-strided" loops -- warp w of the grid handles nodes [32w, 32w+32), then
// jumps by 32 * (warps in the grid).  Loads are coalesced and every lane sees a monotone sequence of
// problem ids (batches are laid out problem after problem), so per-problem reductions run as lane-local
// running accumulators that are flushed on a key change and merged warp-wide (__match_any_sync +
// redux) and block-wide (shared memory) before touching the per-problem atomics.
#pragma once
#include <cooperative_groups.h>

#include "pdp_common.cuh"

namespace cg = cooperative_groups;

struct KArgs {
    pdp_graph g;
    pdp_state s;
    int32_t* trace;      // optional decimation trace: triples (iteration, variable, sign)
    int32_t trace_cap;
    int32_t stagger_c, stagger_v;   // cycles the second CTA of an SM waits at the start of a clause / variable pass
    float dec_fraction;             // pdp_set_decimation_fraction (0: the arg-max rule only)
    // conflict rollback (pdp_set_conflict_rollback): the snapshot of the problems a step decimates, indexed like the state
    // (all null: rollback off)
    struct { float* sol; float* is_sat; uint8_t* av; uint8_t* af; } rb;
    // reinforce (pdp_set_reinforce): the coins, decimation_probability, and whether this run starts at coin 0
    struct { const float* coins; float p; float pi; int32_t fresh; } rf;
};

__device__ __forceinline__ int lane_id() { return threadIdx.x & 31; }
__device__ __forceinline__ int64_t gwarp() { return ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5; }
__device__ __forceinline__ int64_t gwarps() { return ((int64_t)gridDim.x * blockDim.x) >> 5; }
__device__ __forceinline__ int64_t gtid() { return (int64_t)blockIdx.x * blockDim.x + threadIdx.x; }
__device__ __forceinline__ int64_t gthreads() { return (int64_t)gridDim.x * blockDim.x; }

#define WARP_STRIDED(i, N) \
    for (int64_t i##_base = gwarp() * 32, i = i##_base + lane_id(); i##_base < (N); i##_base += gwarps() * 32, i = i##_base + lane_id())

// named barriers (ids 1..15; 0 is __syncthreads): producer / consumer hand-over between warp groups
__device__ __forceinline__ void bar_sync(int id, int n) { asm volatile("bar.sync %0, %1;" ::"r"(id), "r"(n) : "memory"); }
__device__ __forceinline__ void bar_arrive(int id, int n) { asm volatile("bar.arrive %0, %1;" ::"r"(id), "r"(n) : "memory"); }

// ------------------------------------------------------------------------------------------------
// keyed reduction helper.  ACC needs: void reset(); void merge_shfl(unsigned mask) [warp-reduce over
// lanes in `mask`, all of which hold the same key]; void commit(const pdp_state&, int key).
// ------------------------------------------------------------------------------------------------
template <typename ACC>
struct KeyedReducer {
    ACC acc;
    int key;
    __device__ __forceinline__ KeyedReducer() : key(-1) { acc.reset(); }
    // call for every item; commits the running accumulator when the key changes
    __device__ __forceinline__ void touch(const pdp_state& s, int k) {
        if (k != key) {
            if (key >= 0) acc.commit(s, key);
            key = k;
            acc.reset();
        }
    }
    // call once, by ALL threads of the block, outside of divergent code.  Warps whose lanes all hold
    // the same problem merge in registers and hand their partial to a block-level merge in shared
    // memory (one commit per block and problem run: a 1M-variable problem costs ~600 atomics per
    // pass instead of ~10^5); mixed warps commit per lane group.
    __device__ __forceinline__ void finish(const pdp_state& s) {
        __shared__ ACC sm_acc[32];
        __shared__ int sm_key[32];
        const int gthr = blockDim.x, t = threadIdx.x;
        const unsigned m = __match_any_sync(0xffffffffu, key);
        const bool uniform = (m == 0xffffffffu);
        const int warp = t >> 5, nwarp = (gthr + 31) >> 5;
        if (uniform) {
            acc.merge_full();
            if (lane_id() == 0) { sm_acc[warp] = acc; sm_key[warp] = key; }
        } else {
            acc.merge_group(m);
            if (lane_id() == (__ffs(m) - 1) && key >= 0) acc.commit(s, key);
            if (lane_id() == 0) sm_key[warp] = -1;
        }
        __syncthreads();
        if (t == 0) {
            int w = 0;
            while (w < nwarp) {
                const int k = sm_key[w];
                if (k < 0) { ++w; continue; }
                ACC a = sm_acc[w];
                int v = w + 1;
                while (v < nwarp && sm_key[v] == k) { a.merge(sm_acc[v]); ++v; }
                a.commit(s, k);
                w = v;
            }
        }
        __syncthreads();
        key = -1;       // everything has been committed: a later touch() starts from scratch
        acc.reset();
    }
};

__device__ __forceinline__ unsigned long long shfl_xor_u64(unsigned long long v, int o) {
    unsigned lo = __shfl_xor_sync(0xffffffffu, (unsigned)v, o), hi = __shfl_xor_sync(0xffffffffu, (unsigned)(v >> 32), o);
    return ((unsigned long long)hi << 32) | lo;
}

// ------------------------------------------------------------------------------------------------
// accumulators
// ------------------------------------------------------------------------------------------------
struct StatAcc {   // SequentialDecimator statistics: per problem max/min of two smooth-max vectors
    uint32_t mx0, mn0, mx1, mn1, nan, nav;
    __device__ __forceinline__ void reset() { mx0 = 0u; mn0 = 0x7f800000u; mx1 = 0u; mn1 = 0x7f800000u; nan = 0u; nav = 0u; }
    __device__ __forceinline__ void add(float v0, float v1, bool has1, uint32_t act) {
        if (v0 != v0) nan |= 1u; else { uint32_t u = f2u(v0); mx0 = max(mx0, u); mn0 = min(mn0, u); }
        if (has1) { if (v1 != v1) nan |= 2u; else { uint32_t u = f2u(v1); mx1 = max(mx1, u); mn1 = min(mn1, u); } }
        nav += act;
    }
    __device__ __forceinline__ void merge_shfl(unsigned m) {
        mx0 = __reduce_max_sync(m, mx0); mn0 = __reduce_min_sync(m, mn0);
        mx1 = __reduce_max_sync(m, mx1); mn1 = __reduce_min_sync(m, mn1);
        nan = __reduce_or_sync(m, nan); nav = __reduce_add_sync(m, nav);
    }
    __device__ __forceinline__ void merge_full() { merge_shfl(0xffffffffu); }
    __device__ __forceinline__ void merge_group(unsigned m) { merge_shfl(m); }
    __device__ __forceinline__ void merge(const StatAcc& o) {
        mx0 = max(mx0, o.mx0); mn0 = min(mn0, o.mn0); mx1 = max(mx1, o.mx1); mn1 = min(mn1, o.mn1); nan |= o.nan; nav += o.nav;
    }
    __device__ __forceinline__ void commit(const pdp_state& s, int b) const {
        atomicMax(&s.st_max[2 * b], mx0); atomicMin(&s.st_min[2 * b], mn0);
        atomicMax(&s.st_max[2 * b + 1], mx1); atomicMin(&s.st_min[2 * b + 1], mn1);
        if (nan) atomicOr(&s.st_nan[b], nan);
        if (nav) atomicAdd(&s.nav[b], (int)nav);
    }
};

struct CoefAcc {   // decimation coefficients |score| * active: per problem max / min / NaN
    uint32_t mx, mn, nan;
    __device__ __forceinline__ void reset() { mx = 0u; mn = 0x7f800000u; nan = 0u; }
    __device__ __forceinline__ void add(float c) {
        if (c != c) nan = 1u; else { uint32_t u = f2u(c); mx = max(mx, u); mn = min(mn, u); }
    }
    __device__ __forceinline__ void merge_shfl(unsigned m) {
        mx = __reduce_max_sync(m, mx); mn = __reduce_min_sync(m, mn); nan = __reduce_or_sync(m, nan);
    }
    __device__ __forceinline__ void merge_full() { merge_shfl(0xffffffffu); }
    __device__ __forceinline__ void merge_group(unsigned m) { merge_shfl(m); }
    __device__ __forceinline__ void merge(const CoefAcc& o) { mx = max(mx, o.mx); mn = min(mn, o.mn); nan |= o.nan; }
    __device__ __forceinline__ void commit(const pdp_state& s, int b) const {
        atomicMax(&s.c_max[b], mx); atomicMin(&s.c_min[b], mn);
        if (nan) atomicOr(&s.c_nan[b], nan);
    }
};

struct CountAcc {  // integer count into s.n_unsat
    int n;
    __device__ __forceinline__ void reset() { n = 0; }
    __device__ __forceinline__ void merge_shfl(unsigned m) { n = __reduce_add_sync(m, n); }
    __device__ __forceinline__ void merge_full() { merge_shfl(0xffffffffu); }
    __device__ __forceinline__ void merge_group(unsigned m) { merge_shfl(m); }
    __device__ __forceinline__ void merge(const CountAcc& o) { n += o.n; }
    __device__ __forceinline__ void commit(const pdp_state& s, int b) const { if (n) atomicAdd(&s.n_unsat[b], n); }
};

struct EnergyAcc { // integer count into s.energy
    int n;
    __device__ __forceinline__ void reset() { n = 0; }
    __device__ __forceinline__ void merge_shfl(unsigned m) { n = __reduce_add_sync(m, n); }
    __device__ __forceinline__ void merge_full() { merge_shfl(0xffffffffu); }
    __device__ __forceinline__ void merge_group(unsigned m) { merge_shfl(m); }
    __device__ __forceinline__ void merge(const EnergyAcc& o) { n += o.n; }
    __device__ __forceinline__ void commit(const pdp_state& s, int b) const { if (n) atomicAdd(&s.energy[b], n); }
};

// WalkSAT candidate selection (solver.py:453-458): per problem
//   kg = min over variables of (delta, index)            -> first index of the minimum energy delta
//   kr = max over variables of (fl(x+1) bits, ~index)    -> first index of the maximum random key
//   mn / mx = min / max of x (float bits) for the exact handling of min x > 0
struct PickAcc {
    unsigned long long kg, kr;
    uint32_t mn, mx;
    __device__ __forceinline__ void reset() { kg = ~0ull; kr = 0ull; mn = 0x7f800000u; mx = 0u; }
    __device__ __forceinline__ void add(unsigned long long g, unsigned long long r, uint32_t xb) {
        kg = g < kg ? g : kg; kr = r > kr ? r : kr; mn = min(mn, xb); mx = max(mx, xb);
    }
    __device__ __forceinline__ void merge(const PickAcc& o) {
        kg = o.kg < kg ? o.kg : kg; kr = o.kr > kr ? o.kr : kr; mn = min(mn, o.mn); mx = max(mx, o.mx);
    }
    __device__ __forceinline__ void merge_full() {
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) {
            const unsigned long long g = shfl_xor_u64(kg, o), r = shfl_xor_u64(kr, o);
            kg = g < kg ? g : kg; kr = r > kr ? r : kr;
        }
        mn = __reduce_min_sync(0xffffffffu, mn); mx = __reduce_max_sync(0xffffffffu, mx);
    }
    // mixed warp: serialise over the (few) distinct keys; every lane of a group ends with the group's result
    __device__ __forceinline__ void merge_group(unsigned m) {
        mn = __reduce_min_sync(m, mn); mx = __reduce_max_sync(m, mx);
        unsigned todo = m;
        unsigned long long g = kg, r = kr;
        while (todo) {
            const int src = __ffs(todo) - 1;
            const unsigned long long og = __shfl_sync(m, g, src), orr = __shfl_sync(m, r, src);
            kg = og < kg ? og : kg; kr = orr > kr ? orr : kr;
            todo &= todo - 1;
        }
    }
    __device__ __forceinline__ void commit(const pdp_state& s, int b) const {
        atomicMin(&s.ws_key[2 * b], kg); atomicMax(&s.ws_key[2 * b + 1], kr);
        atomicMin(&s.ws_best[2 * b], mn); atomicMax(&s.ws_best[2 * b + 1], mx);
    }
};


// ------------------------------------------------------------------------------------------------
// activity masks.  The edge mask em(e) = active_variable(i(e)) * active_function(a(e)) of the reference
// (solver.py:370-371) is kept as one bit per edge, indexed by the edge's position in each of the two
// message layouts (g.vmask / g.qmask) and set where a node is de-activated: a pass reads the mask bits
// of its region with the same contiguous access as the messages and never gathers the node masks.
// ------------------------------------------------------------------------------------------------
__device__ __forceinline__ void mask_edge(const pdp_graph& g, int vpos, int qpos) {
    atomicOr(&g.vmask[vpos >> 5], 1u << (vpos & 31));
    atomicOr(&g.qmask[qpos >> 5], 1u << (qpos & 31));
}
__device__ __forceinline__ void deactivate_variable(const pdp_graph& g, const pdp_state& s, int i) {
    s.av[i] = 0;
    for (int p = g.var_ptr[i]; p < g.var_ptr[i + 1]; ++p) mask_edge(g, g.p_vpos[p], g.p_qpos[p]);
}

// entry `id` appended to the list whose length is s.ctrl[slot]; a full list raises CTRL_FR_OVER
__device__ __forceinline__ void fr_append(const pdp_state& s, int slot, int32_t* list, int id) {
    const int k = atomicAdd(&s.ctrl[slot], 1);
    if (k < s.fr_cap) list[k] = id; else s.ctrl[CTRL_FR_OVER] = 1;
}
// node `id` put on node list `list` of the frontier closure, once per epoch
__device__ __forceinline__ void fr_push(const pdp_state& s, int list, int32_t* stamp, int id, int epoch) {
    if (atomicExch(&stamp[id], epoch) == epoch) return;
    fr_append(s, CTRL_FR_N + list, s.fr_list[list], id);
}
// Where fixes and clause de-activations queue the nodes they touch.  NoQueue: nowhere (the full scans look at every node).
// ListQueue: the lists of the frontier closure -- the still-active clauses of a fixed variable that its value does not
// satisfy go to clause list clist at epoch epc (unit test; clist < 0: none), the still-active variables of a de-activated
// clause go to variable list vlist at epoch epv (purity test).
struct NoQueue {
    __device__ __forceinline__ void clause(const pdp_state&, int) const {}
    __device__ __forceinline__ void var(const pdp_state&, int) const {}
};
struct ListQueue {
    int clist, epc, vlist, epv;
    __device__ __forceinline__ void clause(const pdp_state& s, int a) const { if (clist >= 0 && s.af[a]) fr_push(s, clist, s.stamp_c, a, epc); }
    __device__ __forceinline__ void var(const pdp_state& s, int j) const { if (s.av[j]) fr_push(s, vlist, s.stamp_v, j, epv); }
};

template <typename Q = NoQueue>
__device__ __forceinline__ void deactivate_clause(const pdp_graph& g, const pdp_state& s, int a, const Q& q = Q()) {
    s.af[a] = 0;
    for (int c = g.cl_ptr[a]; c < g.cl_ptr[a + 1]; ++c) {
        mask_edge(g, cvpos(g, c), cqpos(g, c));
        q.var(s, (int)(g.c_var[c] & PDP_IDX_MASK));
    }
}
// the words change between passes: read around L1
__device__ __forceinline__ bool mbit(const uint32_t* words, int pos) { return (__ldcg(words + (pos >> 5)) >> (pos & 31)) & 1u; }

// variable side of the SP update with the per-variable part hoisted (pi == 0): for one sign s the terms
// 0.5(1+s)P + 0.5(1-s)N, opp and exp(opp) do not depend on the edge.  Same operations, same order as
// sp_var_update_qu.
__device__ __forceinline__ void sp_var_prepare(float P, float N, float s, float& same_base, float& opp, float& O) {
    same_base = 0.5f * (1.f + s) * P + 0.5f * (1.f - s) * N;
    opp = 0.5f * (1.f - s) * P + 0.5f * (1.f + s) * N;   // (the reference's `+ log(1 - 0)` = +0 only turns a -0 into +0: exp is blind to it)
    O = X30(opp);
}
__device__ __forceinline__ float sp_var_finish(float same_base, float opp, float O, float y) {
    const float same = same_base - y;
    const float S = X30(same);
    const float dc = X30(same + opp);
    const float u = S * (1.f - O), v = O * (1.f - S);
    const float total = u + v + dc;
    return pdp_divf(u, total);
}

// the same with the two pi terms of a variable whose external force is the same on all its edges (reinforce on the
// blocked passes): l_same / l_opp = log(max(1 - pi [ext == s], 1e-40)) / log(max(1 - pi [ext == -s], 1e-40)), added in
// the order of sp_var_update
__device__ __forceinline__ void sp_var_prepare_pi(float P, float N, float s, float l_opp, float& same_base, float& opp, float& O) {
    same_base = 0.5f * (1.f + s) * P + 0.5f * (1.f - s) * N;
    opp = 0.5f * (1.f - s) * P + 0.5f * (1.f + s) * N;
    opp += l_opp;
    O = X30(opp);
}
__device__ __forceinline__ float sp_var_finish_pi(float same_base, float l_same, float opp, float O, float y) {
    float same = same_base - y;
    same += l_same;
    const float S = X30(same);
    const float dc = X30(same + opp);
    const float u = S * (1.f - O), v = O * (1.f - S);
    const float total = u + v + dc;
    return pdp_divf(u, total);
}

// ------------------------------------------------------------------------------------------------
// generic passes: thread per node, indexed global accesses.  MODE selects the problems.
// ------------------------------------------------------------------------------------------------
enum { GEN_ALL = 0, GEN_NAN = 1 };
template <int MODE>
__device__ __forceinline__ bool gen_take(const pdp_state& s, int b) {
    if (!s.active[b]) return false;
    return (MODE == GEN_ALL) ? true : (s.nanflag[b] != 0);
}

// clause side: eta'(e) = exp(min(sum_{e' in a(e)} x_e' - x_e, 30)), x = log(max(q_u,1e-40)) * em
// (pdp_propagate.py:166-175).  r = buffer of the previous surveys.
template <int MODE>
__device__ __forceinline__ void gen_clause_side(const KArgs& A, int r, bool use_mask) {
    const pdp_graph& g = A.g; const pdp_state& s = A.s;
    const float* __restrict__ qin = s.qu;
    const float* __restrict__ eold = s.eta[r];
    float* __restrict__ eout = s.eta[r ^ 1];
    WARP_STRIDED(a, g.F) {
        if (a >= g.F) continue;
        const int b = g.bfm[a];
        if (!gen_take<MODE>(s, b)) continue;
        const bool um = use_mask && s.masked[b];
        // the reference blends `mask*new + (1-mask)*old` arithmetically, so a NaN message is sticky
        // (0*NaN); problems that have produced a NaN re-read the old value
        const bool sticky = s.nanflag[b] != 0;
        bool made_nan = false;
        const int beg = g.cl_ptr[a], end = g.cl_ptr[a + 1];
        float tot = 0.f;
        for (int c = beg; c < end; ++c) {
            const int qp = cqpos(g, c);
            float v = L40(qin[qp]);
            if (um && mbit(g.qmask, qp)) v = v * 0.f;
            tot += v;
        }
        for (int c = beg; c < end; ++c) {
            const int qp = cqpos(g, c);
            float v = L40(qin[qp]);
            if (um && mbit(g.qmask, qp)) v = v * 0.f;
            const int pos = cvpos(g, c);
            float nv = X30(tot - v);
            if (sticky) { const float ov = eold[pos]; if (ov != ov) nv = ov; }
            made_nan |= (nv != nv);
            eout[pos] = nv;
        }
        if (made_nan && !sticky) s.nanpend[b] = 1;
    }
}

// variable side (pdp_propagate.py:184-218): q(t) from eta[r], written in place
template <int MODE, bool FULL>
__device__ __forceinline__ void gen_var_side(const KArgs& A, int r, bool use_mask, float pi) {
    const pdp_graph& g = A.g; const pdp_state& s = A.s;
    const float* __restrict__ ein = s.eta[r];
    WARP_STRIDED(i, g.V) {
        if (i >= g.V) continue;
        const int b = g.bvm[i];
        if (!gen_take<MODE>(s, b)) continue;
        const bool um = use_mask && s.masked[b];
        const int beg = g.var_ptr[i], end = g.var_ptr[i + 1];
        const bool sticky = s.nanflag[b] != 0;
        bool made_nan = false;
        float P = 0.f, N = 0.f;
        for (int p = beg; p < end; ++p) {
            const int vp = g.p_vpos[p];
            const bool neg = (g.v_cedge[p] & PDP_SIGN_BIT) != 0u;
            float y = L40_1m(ein[vp]);
            if (um && mbit(g.vmask, vp)) y = y * 0.f;
            // the reference's pos/neg incidence matrices hold explicit zeros: 0*y keeps NaN alive
            P += (neg ? 0.f : 1.f) * y;
            N += (neg ? 1.f : 0.f) * y;
        }
        for (int p = beg; p < end; ++p) {
            const int vp = g.p_vpos[p];
            float y = L40_1m(ein[vp]);
            if (um && mbit(g.vmask, vp)) y = y * 0.f;
            const float sg = (g.v_cedge[p] & PDP_SIGN_BIT) ? -1.f : 1.f;
            const int qp = g.p_qpos[p];
            if (FULL || pi != 0.f) {
                float u, v, d;
                sp_var_update(P, N, y, sg, s.ext[p], pi, u, v, d);
                if (sticky) {
                    const float ou = s.qu[qp]; if (ou != ou) u = ou;
                    if (FULL) { const float ov = s.qs[qp], od = s.qd[qp]; if (ov != ov) v = ov; if (od != od) d = od; }
                }
                made_nan |= (u != u);
                s.qu[qp] = u;
                if (FULL) { s.qs[qp] = v; s.qd[qp] = d; }
            } else {
                float u = sp_var_update_qu(P, N, y, sg);
                if (sticky) { const float ou = s.qu[qp]; if (ou != ou) u = ou; }
                made_nan |= (u != u);
                s.qu[qp] = u;
            }
        }
        if (made_nan && !sticky) s.nanpend[b] = 1;
    }
}

// decimator statistics (pdp_decimate.py:127-143, util.py:282-286): per variable smooth-max of the new
// surveys and of |eta_prev - eta_new| * edge_mask, times active_variables; per problem max / min.
// w = buffer holding the new surveys.
template <int MODE>
__device__ __forceinline__ void gen_stats(const KArgs& A, int w, bool has_prev, bool em_set) {
    const pdp_graph& g = A.g; const pdp_state& s = A.s;
    const float* __restrict__ en = s.eta[w];
    const float* __restrict__ eo = s.eta[w ^ 1];
    KeyedReducer<StatAcc> red;
    WARP_STRIDED(i, g.V) {
        if (i >= g.V) continue;
        const int b = g.bvm[i];
        if (!gen_take<MODE>(s, b)) continue;
        red.touch(s, b);
        const int beg = g.var_ptr[i], end = g.var_ptr[i + 1];
        const uint32_t act = s.av[i];
        const bool um = em_set && s.masked[b];
        float n0 = 0.f, d0 = 0.f, n1 = 0.f, d1 = 0.f;
        for (int p = beg; p < end; ++p) {
            const int pos = g.p_vpos[p];
            const float v = en[pos];
            const float c = X30S(v);
            n0 += v * c; d0 += c;
            if (has_prev) {
                float d = fabsf(eo[pos] - v);
                if (um && mbit(g.vmask, pos)) d = d * 0.f;
                const float cd = X30S(d);
                n1 += d * cd; d1 += cd;
            }
        }
        const float sm0 = pdp_divs(n0, tmaxf(d0, 1.0f)) * (float)act;
        const float sm1 = pdp_divs(n1, tmaxf(d1, 1.0f)) * (float)act;
        red.acc.add(sm0, sm1, has_prev, act);
    }
    red.finish(s);
}

#include "pdp_sweep.cuh"

// ------------------------------------------------------------------------------------------------
// SurveyScorer over the converged problems (pdp_predict.py:155-192) + coefficient statistics
// ------------------------------------------------------------------------------------------------
__device__ __forceinline__ float score_variable(const pdp_graph& g, const pdp_state& s, const float* __restrict__ eta,
                                                int i, float pi) {
    const int beg = g.var_ptr[i], end = g.var_ptr[i + 1];
    float extsum = 0.f, ps = 0.f, ns = 0.f, as = 0.f;
    for (int p = beg; p < end; ++p) {
        extsum += s.ext[p];
        const float f = L10(1.f - eta[g.p_vpos[p]]) * (float)s.af[g.v_cls[p]];
        const bool neg = (g.v_cedge[p] & PDP_SIGN_BIT) != 0u;
        ps += (neg ? 0.f : 1.f) * f;
        ns += (neg ? 1.f : 0.f) * f;
        as += f;
    }
    return sp_score_tail(ps, ns, as, sgnf(extsum), pi);
}

// A batch of a few large problems: the grid walks the node range of each flagged problem (no per-node problem
// look-up, no dependent loads, one block-level merge per problem) instead of scanning every node of the batch.
#define PDP_RANGE_SCAN_MAX_B 64
__device__ __forceinline__ bool range_scans(const pdp_graph& g) { return g.contiguous_problems && g.B <= PDP_RANGE_SCAN_MAX_B; }

__device__ __forceinline__ void score_phase(const KArgs& A, int w, float pi) {
    const pdp_graph& g = A.g; const pdp_state& s = A.s;
    KeyedReducer<CoefAcc> red;
    if (range_scans(g)) {
        for (int b = 0; b < (int)g.B; ++b) {
            if (!s.conv[b]) continue;
            const int v1 = g.prob_vptr[b + 1];
            const bool have = s.have_score[b] != 0;
            red.touch(s, b);
            if (have) {
#pragma unroll 4
                for (int i = g.prob_vptr[b] + (int)gtid(); i < v1; i += (int)gthreads())
                    red.acc.add(fabsf(s.score[i]) * (float)s.av[i]);
            } else {
                for (int i = g.prob_vptr[b] + (int)gtid(); i < v1; i += (int)gthreads()) {
                    const float sc = score_variable(g, s, s.eta[w], i, pi);
                    s.score[i] = sc;
                    red.acc.add(fabsf(sc) * (float)s.av[i]);
                }
            }
            red.finish(s);
        }
        return;
    }
    WARP_STRIDED(i, g.V) {
        if (i >= g.V) continue;
        const int b = g.bvm[i];
        if (!s.conv[b]) continue;
        red.touch(s, b);
        float sc;
        if (s.have_score[b]) sc = s.score[i];     // written by this iteration's variable pass (ph_var_score)
        else { sc = score_variable(g, s, s.eta[w], (int)i, pi); s.score[i] = sc; }
        red.acc.add(fabsf(sc) * (float)s.av[i]);
    }
    red.finish(s);
}

// decimation coefficient c_i = |score_i| * active_i of the fused loop (pdp_decimate.py:153)
struct CoefScore {
    const pdp_state& s;
    __device__ __forceinline__ float operator()(int64_t i) const { return fabsf(s.score[i]) * (float)s.av[i]; }
};
// coefficients handed in by the caller (pdp_decimation_select)
struct CoefGiven {
    const float* c;
    __device__ __forceinline__ float operator()(int64_t i) const { return c[i]; }
};

// first index attaining max of fl(fl(c - min) + 1)  (util.py:257-265)
template <typename CF>
__device__ __forceinline__ void argmax_phase(const KArgs& A, const CF& coef) {
    const pdp_graph& g = A.g; const pdp_state& s = A.s;
    if (range_scans(g)) {
        for (int b = 0; b < (int)g.B; ++b) {
            if (!s.conv[b] || s.c_nan[b]) continue;
            const float m = u2f(s.c_min[b]);
            const float kmax = argmax_key(u2f(s.c_max[b]), m);
            const int v1 = g.prob_vptr[b + 1];
#pragma unroll 4
            for (int i = g.prob_vptr[b] + (int)gtid(); i < v1; i += (int)gthreads()) {
                const float c = coef(i);
                if (argmax_key(c, m) == kmax) atomicMin(&s.arg_idx[b], i);
            }
        }
        return;
    }
    WARP_STRIDED(i, g.V) {
        if (i >= g.V) continue;
        const int b = g.bvm[i];
        if (!s.conv[b] || s.c_nan[b]) continue;
        const float m = u2f(s.c_min[b]);
        const float kmax = argmax_key(u2f(s.c_max[b]), m);
        const float c = coef(i);
        if (argmax_key(c, m) == kmax) atomicMin(&s.arg_idx[b], (int)i);
    }
}

// fixing one variable (the per-variable form of _set_variable_core, solver.py:205-226): clauses
// holding a now-true occurrence are de-activated, the variable is de-activated, solution updated.
// STRIDE 1: by one thread; 32: by the lanes of a warp, over the variable's edges, once all of them have read av[i] (the
// decimation fix of a large problem: one thread walking its ~40 dependent global updates was 0.4 ms)
template <int STRIDE = 1, typename Q = NoQueue>
__device__ __forceinline__ void fix_variable(const pdp_graph& g, const pdp_state& s, int i, float sg, const Q& q = Q()) {
    const int lane = STRIDE == 1 ? 0 : lane_id();
    for (int p = g.var_ptr[i] + lane; p < g.var_ptr[i + 1]; p += STRIDE) {
        const float lit = (g.v_cedge[p] & PDP_SIGN_BIT) ? -1.f : 1.f;
        const int a = g.v_cls[p];
        if (lit * sg > 0.f) { if (s.af[a]) deactivate_clause(g, s, a, q); }
        else q.clause(s, a);
        mask_edge(g, g.p_vpos[p], g.p_qpos[p]);
    }
    if (lane == 0) { s.av[i] = 0; s.sol[i] = (sg + 1.f) / 2.0f; }
}

// one event (iteration, variable, sign) of the optional decimation trace
__device__ __forceinline__ void record_fix(const KArgs& A, int iter, int i, float sg) {
    if (!A.trace) return;
    const int k = atomicAdd(&A.s.ctrl[CTRL_TRACE_LEN], 1);
    if (k < A.trace_cap) { A.trace[3 * k] = iter; A.trace[3 * k + 1] = i; A.trace[3 * k + 2] = (int)sg; }
}

// ------------------------------------------------------------------------------------------------
// Conflict rollback (pdp_set_conflict_rollback).  A decimation step of problem b with K_b >= 2 and a clear conflict bit
// first copies b's node masks, solution and is_sat to the caller's snapshot buffer (one byte per node mask, indexed like the
// state: neighbouring problems never write the same byte, so their copies need no atomics).  When the closure after the fix
// sets b's conflict bit, the nodes go back to the snapshot and the edge-mask bits of b's edges are rebuilt from the restored
// node masks; the messages, previous surveys and counters are not touched, the step changed none of them.
// A restored state is one the library itself produced and closed under UP + peeling before this step: the precondition of
// the frontier closure (CTRL_CLOSED) and that of the CNF count (CTRL_NATIVE, only the library changed the masks) still hold.
// ------------------------------------------------------------------------------------------------
// (the conflict marking of the grid-wide closure) b's top-K step conflicted: flag it for rb_restore_grid
__device__ __forceinline__ void rb_mark(const KArgs& A, int b) {
    const pdp_state& s = A.s;
    if (A.rb.av && s.rb_snap[b]) { s.rb_snap[b] = 2; s.ctrl[CTRL_RB] = 1; }
}
__device__ __forceinline__ void rb_save_var(const KArgs& A, int i) { A.rb.av[i] = A.s.av[i]; A.rb.sol[i] = A.s.sol[i]; }
__device__ __forceinline__ void rb_save_clause(const KArgs& A, int a) { A.rb.af[a] = A.s.af[a]; }
// one edge-mask bit; atomic because a mask word holds edges of other nodes and problems
__device__ __forceinline__ void rb_edge_bit(uint32_t* words, int pos, bool masked) {
    const uint32_t bit = 1u << (pos & 31);
    const bool now = (__ldcg(words + (pos >> 5)) & bit) != 0u;
    if (masked && !now) atomicOr(words + (pos >> 5), bit);
    else if (!masked && now) atomicAnd(words + (pos >> 5), ~bit);
}
// variable i back to the snapshot, with the mask bits of its edges (taken from the snapshot's masks, so the clause restores
// need not be complete)
__device__ __forceinline__ void rb_restore_var(const KArgs& A, int i) {
    const pdp_graph& g = A.g; const pdp_state& s = A.s;
    const uint8_t v = A.rb.av[i];
    s.av[i] = v;
    s.sol[i] = A.rb.sol[i];
    for (int p = g.var_ptr[i]; p < g.var_ptr[i + 1]; ++p) {
        const bool masked = !(v && A.rb.af[g.v_cls[p]]);
        rb_edge_bit(g.vmask, g.p_vpos[p], masked);
        rb_edge_bit(g.qmask, g.p_qpos[p], masked);
    }
}
__device__ __forceinline__ void rb_restore_clause(const KArgs& A, int a) { A.s.af[a] = A.rb.af[a]; }
// the per-problem part of a rollback (one thread)
__device__ __forceinline__ void rb_commit(const KArgs& A, int b, int iter) {
    const pdp_state& s = A.s;
    s.is_sat[b] = A.rb.is_sat[b];
    s.flags[b] = (s.flags[b] & ~PDP_FLAG_UP_CONFLICT) | PDP_FLAG_ROLLED_BACK;
    s.rb_h[b] += 1;
    s.rb_count[b] += 1;
    s.rb_last[b] = iter;
}

// ------------------------------------------------------------------------------------------------
// clause and variable tests of the closures and the CNF check.  A clause -> variable CSR word W is the variable's index
// with the literal's sign in the top bit: 32 bits in g.c_var, 16 bits (local indices) in the shared-memory tier.
// ------------------------------------------------------------------------------------------------
// literal of sign sgn (+-1) true under the solution value p (SatCNFEvaluator, util.py:210-236)
__device__ __forceinline__ bool literal_true(float sgn, float p) {
    float ev = sgn * p;
    ev = ev + (1.f - sgn) / 2.f;
    return ev > 0.5f;
}
// clause [beg, end) of the CSR holds a true literal under sol
template <typename W>
__device__ __forceinline__ bool clause_satisfied(const W* cvar, int beg, int end, const float* sol) {
    constexpr uint32_t sign = 1u << (8 * sizeof(W) - 1);
    for (int c = beg; c < end; ++c) {
        const uint32_t w = cvar[c];
        if (literal_true((w & sign) ? -1.f : 1.f, sol[w & (sign - 1u)])) return true;
    }
    return false;
}
// clause [beg, end) of the CSR has exactly one active variable: j, and whether it occurs negated
template <typename W>
__device__ __forceinline__ bool clause_unit(const W* cvar, int beg, int end, const uint8_t* av, int& j, bool& neg) {
    constexpr uint32_t sign = 1u << (8 * sizeof(W) - 1);
    int deg = 0; uint32_t hit = 0;
    for (int c = beg; c < end; ++c) {
        const uint32_t w = cvar[c];
        if (av[w & (sign - 1u)]) { ++deg; hit = w; }
    }
    j = (int)(hit & (sign - 1u)); neg = (hit & sign) != 0u;
    return deg == 1;
}
// variable i occurs in the active clauses with one sign only, or in none: val = the solution value peeling gives it
__device__ __forceinline__ bool var_pure(const pdp_graph& g, const uint8_t* af, int i, float& val) {
    int deg = 0, sdeg = 0;
    for (int p = g.var_ptr[i]; p < g.var_ptr[i + 1]; ++p)
        if (af[g.v_cls[p]]) { ++deg; sdeg += (g.v_cedge[p] & PDP_SIGN_BIT) ? -1 : 1; }
    val = ((sdeg > 0 ? 1.f : (sdeg < 0 ? -1.f : 0.f)) + 1.f) / 2.0f;
    return deg == abs(sdeg);
}

// ------------------------------------------------------------------------------------------------
// Grid-wide closure: unit propagation rounds, then pure-literal peeling rounds, to the fixed point of the dirty problems
// (solver.py:180-273), for large problems, batch replication, simplify() and set_variables().  One body, closure_rounds,
// runs the synchronous rounds -- every phase reads only what the barrier before it published -- over a node source: the
// nodes a round looks at, and the queue its fixes and de-activations put the nodes they touch on.
//  * FullScan: every node (of the dirty problems); queues nothing, never overflows.  The closure of simplify() and set_variables(), the
//    fallback of the frontier, and the reference of the tests (flags bit 2).
//  * Frontier: lists of the nodes touched since the round before.  Once every problem is closed under unit propagation
//    and peeling (after simplify()), fixing a variable can only create unit clauses among the clauses that hold a
//    variable de-activated in the previous round, and pure literals among the variables of clauses de-activated since:
//    the same rounds over those lists instead of over all F clauses and V variables (8.9 -> 1.9 ms per decimation
//    iteration at 8 x n = 1 M, where a round's full scan gathers 100 M node flags to find a dozen nodes).
// ------------------------------------------------------------------------------------------------
struct FullScan {
    template <typename Fn> __device__ __forceinline__ void clauses(const KArgs& A, int, Fn fn) const {
        WARP_STRIDED(a, A.g.F) { if (a < A.g.F) fn((int)a); }
    }
    template <typename Fn> __device__ __forceinline__ void units(const KArgs& A, int, Fn fn) const {
        WARP_STRIDED(i, A.g.V) { if (i < A.g.V) fn((int)i); }
    }
    template <typename Fn> __device__ __forceinline__ void vars(const KArgs& A, int round, Fn fn) const { units(A, round, fn); }
    __device__ __forceinline__ void unit(const pdp_state&, int, int) const {}
    __device__ __forceinline__ NoQueue up_queue(int) const { return {}; }
    __device__ __forceinline__ NoQueue peel_queue(int) const { return {}; }
    __device__ __forceinline__ bool up_round(const pdp_state&, int) const { return true; }
    __device__ __forceinline__ bool peel_round(const pdp_state&, int) const { return true; }
};

// Ping-pong lists, entries unique per epoch (stamps):
//   clause lists 0/1 (by UP round)    : clauses to test for unit-ness
//   variable lists 2/3 (by peel round): variables to test for purity; list 2 is filled during the whole UP stage
//   unit lists 0/1 (by UP round)      : variables some unit clause of the round points at (at most one per clause of the
//                                       round's list: they cannot overflow)
template <typename Fn>
__device__ __forceinline__ void fr_each(const pdp_state& s, int slot, const int32_t* list, Fn fn) {
    const int n = s.ctrl[slot] < s.fr_cap ? s.ctrl[slot] : s.fr_cap;
    WARP_STRIDED(x, n) { if (x < n) fn(list[x]); }
}
struct Frontier {
    int epc, epv;   // epochs of the clause list and of the variable list the current round reads
    template <typename Fn> __device__ __forceinline__ void clauses(const KArgs& A, int round, Fn fn) const {
        fr_each(A.s, CTRL_FR_N + (round & 1), A.s.fr_list[round & 1], fn);
    }
    template <typename Fn> __device__ __forceinline__ void units(const KArgs& A, int round, Fn fn) const {
        fr_each(A.s, CTRL_FR_NU + (round & 1), A.s.fr_unit[round & 1], fn);
    }
    template <typename Fn> __device__ __forceinline__ void vars(const KArgs& A, int round, Fn fn) const {
        fr_each(A.s, CTRL_FR_N + 2 + (round & 1), A.s.fr_list[2 + (round & 1)], fn);
    }
    __device__ __forceinline__ void unit(const pdp_state& s, int round, int j) const {
        fr_append(s, CTRL_FR_NU + (round & 1), s.fr_unit[round & 1], j);
    }
    // UP round r queues clauses for round r + 1 and variables for peel round 0; peel round r queues variables for
    // peel round r + 1
    __device__ __forceinline__ ListQueue up_queue(int round) const { return {(round & 1) ^ 1, epc + 1, 2, epv}; }
    __device__ __forceinline__ ListQueue peel_queue(int round) const { return {-1, 0, 2 + ((round & 1) ^ 1), epv + 1}; }
    // the top of a round, by all threads: the epoch of the round's list; thread 0 empties the lists the round fills.
    // False when a list has overflowed (uniform: written before the last barrier).
    __device__ __forceinline__ bool up_round(const pdp_state& s, int round) {
        if (round > 0) ++epc;
        if (s.ctrl[CTRL_FR_OVER]) return false;
        if (gtid() == 0) { s.ctrl[CTRL_FR_N + ((round & 1) ^ 1)] = 0; s.ctrl[CTRL_FR_NU + ((round & 1) ^ 1)] = 0; }
        return true;
    }
    __device__ __forceinline__ bool peel_round(const pdp_state& s, int round) {
        if (round > 0) ++epv;
        if (s.ctrl[CTRL_FR_OVER]) return false;
        if (gtid() == 0) s.ctrl[CTRL_FR_N + 2 + ((round & 1) ^ 1)] = 0;
        return true;
    }
};

// unit propagation round (solver.py:228-273), split at its data dependencies
template <typename Src>
__device__ __forceinline__ void find_units(const KArgs& A, const Src& src, int round, int flag_slot) {
    const pdp_graph& g = A.g; const pdp_state& s = A.s;
    src.clauses(A, round, [&](int a) {
        if (!s.af[a] || !s.dirty[g.bfm[a]]) return;
        int j; bool neg;
        if (!clause_unit(g.c_var, g.cl_ptr[a], g.cl_ptr[a + 1], s.av, j, neg)) return;
        s.single[a] = 1;
        if (atomicAdd(&s.up_cnt[j], 1) == 0) src.unit(s, round, j);
        atomicAdd(&s.up_ev[j], neg ? -1 : 1);
        s.ctrl[flag_slot] = 1;
    });
}

// a problem's first conflict raises CTRL_UP_WIPE: one conflict may mean a wipe
template <typename Src>
__device__ __forceinline__ void find_conflicts(const KArgs& A, const Src& src, int round) {
    const pdp_graph& g = A.g; const pdp_state& s = A.s;
    src.units(A, round, [&](int i) {
        const int cnt = s.up_cnt[i];
        if (cnt > 0 && abs(s.up_ev[i]) != cnt && atomicAdd(&s.conflicts[g.bvm[i]], 1) == 0) s.ctrl[CTRL_UP_WIPE] = 1;
    });
}

// quirk kept from the reference (solver.py:257,261): the problem is wiped only when its conflict COUNT equals exactly one;
// the wipe scans the whole batch (rare).  RB: conflict rollback of the fused loop's grid-wide step (rb_mark)
template <bool RB, typename Src>
__device__ __forceinline__ void apply_conflicts(const KArgs& A, const Src& src, int round) {
    const pdp_graph& g = A.g; const pdp_state& s = A.s;
    const auto q = src.up_queue(round);
    src.clauses(A, round, [&](int a) {
        if (s.single[a]) { deactivate_clause(g, s, a, q); s.single[a] = 0; s.masked[g.bfm[a]] = 1; }
    });
    if (s.ctrl[CTRL_UP_WIPE]) {
        const int64_t n = g.V > g.F ? g.V : g.F;
        WARP_STRIDED(i, n) {
            if (i < g.F && s.af[i] && !s.single[i] && s.conflicts[g.bfm[i]] == 1) deactivate_clause(g, s, (int)i);
            if (i < g.V && s.av[i] && s.conflicts[g.bvm[i]] == 1) deactivate_variable(g, s, (int)i);
        }
    }
    WARP_STRIDED(b, g.B) {
        if (b < g.B && s.conflicts[b] >= 1) { s.is_sat[b] = 0.f; s.flags[b] |= PDP_FLAG_UP_CONFLICT; s.masked[b] = 1; if (RB) rb_mark(A, (int)b); }
    }
}

template <typename Src>
__device__ __forceinline__ void assign_units(const KArgs& A, const Src& src, int round) {
    const pdp_graph& g = A.g; const pdp_state& s = A.s;
    const auto q = src.up_queue(round);
    src.units(A, round, [&](int i) {
        const int cnt = s.up_cnt[i];
        if (cnt > 0) {
            const int ev = s.up_ev[i];
            s.up_cnt[i] = 0; s.up_ev[i] = 0;
            if (s.av[i] && abs(ev) == cnt) fix_variable(g, s, i, ev > 0 ? 1.f : -1.f, q);
        }
    });
    WARP_STRIDED(b, g.B) { if (b < g.B) s.conflicts[b] = 0; }
    if (gtid() == 0) s.ctrl[CTRL_UP_WIPE] = 0;
}

// pure-literal peeling round (solver.py:180-203)
template <typename Src>
__device__ __forceinline__ void peel_find(const KArgs& A, const Src& src, int round, int flag_slot) {
    const pdp_graph& g = A.g; const pdp_state& s = A.s;
    src.vars(A, round, [&](int i) {
        if (!s.av[i] || !s.dirty[g.bvm[i]]) return;
        float val;
        if (var_pure(g, s.af, i, val)) { s.pure[i] = 1; s.sol[i] = val; s.ctrl[flag_slot] = 1; }
    });
}

// a pure variable is fixed to the value the round gave it: every active clause holding it is satisfied (none holds it:
// sol 0.5, sign 0, and it only leaves the problem), so the fix queues no clause
template <typename Src>
__device__ __forceinline__ void peel_fix(const KArgs& A, const Src& src, int round) {
    const pdp_graph& g = A.g; const pdp_state& s = A.s;
    const auto q = src.peel_queue(round);
    src.vars(A, round, [&](int i) {
        if (!s.pure[i]) return;
        s.pure[i] = 0;
        fix_variable(g, s, i, 2.f * s.sol[i] - 1.f, q);
        s.masked[g.bvm[i]] = 1;
    });
}

// The rounds over node source src, by ALL threads of the cooperative grid; false when the source's lists overflowed (at
// the top of a round: the per-round scratch is clean).  Flag slots alternate by round parity so a flag is never reset
// while it can still be read; UP and peel use disjoint slots so a thread that has left one loop can never disturb a flag
// another thread is still reading.  Every flag slot is zero again after a true return.
template <bool RB, typename Src>
__device__ __forceinline__ bool closure_rounds(const KArgs& A, cg::grid_group& grid, Src& src) {
    const pdp_state& s = A.s;
    for (int round = 0;; ++round) {   // solver.py:234-273
        const int slot = CTRL_FLAG_A + (round & 1);
        if (!src.up_round(s, round)) return false;
        find_units(A, src, round, slot);
        if (gtid() == 0) s.ctrl[CTRL_FLAG_A + ((round + 1) & 1)] = 0;
        grid.sync();
        if (!s.ctrl[slot]) break;
        find_conflicts(A, src, round);
        grid.sync();
        apply_conflicts<RB>(A, src, round);
        grid.sync();
        assign_units(A, src, round);
        grid.sync();
    }
    for (int round = 0;; ++round) {   // solver.py:188-203
        const int slot = CTRL_FLAG_C + (round & 1);
        if (!src.peel_round(s, round)) return false;
        peel_find(A, src, round, slot);
        if (gtid() == 0) s.ctrl[CTRL_FLAG_C + ((round + 1) & 1)] = 0;
        grid.sync();
        if (!s.ctrl[slot]) break;
        peel_fix(A, src, round);
        grid.sync();
    }
    return true;
}

template <bool RB = false>
__device__ PDP_COLD void closure(const KArgs& A, cg::grid_group& grid) {
    FullScan src;
    closure_rounds<RB>(A, grid, src);
}

// the queue of the decimation fixes closure_frontier starts from: clause list 0 and variable list 2
__device__ __forceinline__ ListQueue frontier_queue(const pdp_state& s) { return {0, s.ctrl[CTRL_FR_EPC], 2, s.ctrl[CTRL_FR_EPV]}; }

// after those fixes and a grid barrier.  A list that overflows sends the rest of the closure through the full scans.
template <bool RB = false>
__device__ PDP_COLD void closure_frontier(const KArgs& A, cg::grid_group& grid) {
    const pdp_state& s = A.s;
    Frontier src{s.ctrl[CTRL_FR_EPC], s.ctrl[CTRL_FR_EPV]};
    const bool closed = closure_rounds<RB>(A, grid, src);
    grid.sync();
    if (gtid() == 0) {
        s.ctrl[CTRL_FR_EPC] = src.epc + 1; s.ctrl[CTRL_FR_EPV] = src.epv + 1;
        for (int i = 0; i < 4; ++i) s.ctrl[CTRL_FR_N + i] = 0;
        s.ctrl[CTRL_FR_NU] = 0; s.ctrl[CTRL_FR_NU + 1] = 0; s.ctrl[CTRL_FR_OVER] = 0;
    }
    if (!closed) {
        if (gtid() == 0) { s.ctrl[CTRL_FLAG_A] = 0; s.ctrl[CTRL_FLAG_A + 1] = 0; s.ctrl[CTRL_FLAG_C] = 0; s.ctrl[CTRL_FLAG_C + 1] = 0; }
        grid.sync();
        closure<RB>(A, grid);
    }
}

// ------------------------------------------------------------------------------------------------
// Fractional decimation (SP-inspired decimation, Braunstein, Mezard, Zecchina 2005): the rule of pdp_decimate.py:152-171
// fixes the arg-max variable of every selected problem; with a fraction f > 0 a problem b with A_b active variables takes
// K_b = max(1, floor(f * A_b)) variables per step.  K_b == 1 keeps the arg-max rule above unchanged.  K_b >= 2 takes the
// first min(K_b, #candidates) active variables with c > 0 ordered by c descending, then index ascending: a per-problem
// radix select, 8 bits per pass from the top, on the unique 64-bit key (float bits of c) << 32 | (0xFFFFFFFF - index)
// (c >= 0: its bits order like unsigned integers).  A pass stops refining a problem as soon as the bucket holding the K-th
// key is taken whole; the rule that remains is (key >> sel_sh) >= sel_pref.
// ------------------------------------------------------------------------------------------------
__device__ __forceinline__ unsigned long long sel_key(float c, int64_t i) {
    return ((unsigned long long)__float_as_uint(c) << 32) | (unsigned long long)(0xFFFFFFFFu - (uint32_t)i);
}
// K_b in double from the fp32 fraction, halved h times (conflict rollback)
__device__ __forceinline__ int sel_k(float f, int nav, int h) {
    const double k = floor((double)f * (double)nav);
    const int64_t q = (int64_t)k >> (h < 62 ? h : 62);
    return q < 1 ? 1 : (int)q;
}
// warp-aggregated histogram increment (all 32 lanes call it): lanes hitting the same bin add once
__device__ __forceinline__ void sel_count(uint32_t* bin, bool pred) {
    const unsigned long long a = pred ? (unsigned long long)(uintptr_t)bin : 0ull;
    const unsigned m = __match_any_sync(0xffffffffu, a);
    if (pred && lane_id() == __ffs(m) - 1) atomicAdd(bin, (uint32_t)__popc(m));
}
// histogram of one variable: `first` = pass 0 (every candidate, plus the active-variable count); otherwise candidates
// whose key agrees with the bits fixed so far.  All lanes call it; `valid` = the variable belongs to a selecting problem.
__device__ __forceinline__ void sel_hist_var(const pdp_state& s, bool valid, int b, int64_t i, float c, bool act, bool first) {
    uint32_t* h = s.sel_hist + (size_t)(valid ? b : 0) * PDP_SEL_BINS;
    const bool cand = valid && act && c > 0.f;
    const unsigned long long key = sel_key(c, i);
    int sh = 56;
    bool in = cand;
    if (!first && cand) { sh = s.sel_sh[b]; in = (key >> (sh + 8)) == s.sel_pref[b]; }
    if (first) sel_count(h + 256, valid && act);
    sel_count(h + (int)((key >> sh) & 255u), in);
}
// is variable i (coefficient c, active) taken by the final rule of its problem
__device__ __forceinline__ bool sel_taken(const pdp_state& s, int b, int64_t i, float c, bool act) {
    return act && c > 0.f && (sel_key(c, i) >> s.sel_sh[b]) >= s.sel_pref[b];
}

// one warp, after a histogram pass of problem b: picks the digit that holds the K-th key, clears the histogram, updates the
// problem's state.  first: K_b from the active-variable count (halve: shifted right by the problem's rb_h); a problem with
// K_b == 1 leaves (sel_need = -1) for the arg-max rule.  Returns -1 (arg-max rule), 0 (final rule) or 1 (another pass), the
// same in every lane.
__device__ __forceinline__ int sel_decide(const pdp_state& s, int b, float frac, bool first, bool halve) {
    uint32_t* h = s.sel_hist + (size_t)b * PDP_SEL_BINS;
    const int lane = lane_id();
    uint32_t v[8], tot = 0;
#pragma unroll
    for (int k = 0; k < 8; ++k) { v[k] = h[8 * lane + k]; tot += v[k]; }
    int need, sh;
    unsigned long long pref;
    const int nav = first ? (int)h[256] : 0;
    __syncwarp();
#pragma unroll
    for (int k = 0; k < 8; ++k) h[8 * lane + k] = 0u;
    if (first && lane == 0) h[256] = 0u;
    // inclusive suffix sums over the lanes: keys in bins >= 8 * lane
    uint32_t suf = tot;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) { const uint32_t y = __shfl_down_sync(0xffffffffu, suf, o); if (lane + o < 32) suf += y; }
    if (first) {
        const int K = sel_k(frac, nav, halve ? s.rb_h[b] : 0);
        const uint32_t ncand = __shfl_sync(0xffffffffu, suf, 0);
        if (K < 2) { if (lane == 0) s.sel_need[b] = -1; return -1; }
        if (ncand <= (uint32_t)K) {   // every candidate is taken
            if (lane == 0) { s.sel_need[b] = 0; s.sel_sh[b] = 0; s.sel_pref[b] = 0ull; }
            return 0;
        }
        need = K; sh = 56; pref = 0ull;
    } else {
        need = s.sel_need[b]; sh = s.sel_sh[b]; pref = s.sel_pref[b];
    }
    // the lane whose bins hold the need-th key from the top, then the bin inside it
    const uint32_t above_lane = suf - tot;
    const bool mine = above_lane < (uint32_t)need && suf >= (uint32_t)need;
    const int src = __ffs(__ballot_sync(0xffffffffu, mine)) - 1;
    int d = 0; uint32_t above = 0, cnt = 0;
    if (mine) {
        uint32_t cum = above_lane;
#pragma unroll
        for (int k = 7; k >= 0; --k) {
            if (cum + v[k] >= (uint32_t)need) { d = 8 * lane + k; above = cum; cnt = v[k]; break; }
            cum += v[k];
        }
    }
    d = __shfl_sync(0xffffffffu, d, src); above = __shfl_sync(0xffffffffu, above, src); cnt = __shfl_sync(0xffffffffu, cnt, src);
    pref = (pref << 8) | (unsigned long long)d;
    const bool done = cnt == (uint32_t)need - above;   // the bucket is taken whole (always true at shift 0: keys are unique)
    if (lane == 0) {
        s.sel_pref[b] = pref;
        if (done) { s.sel_need[b] = 0; s.sel_sh[b] = sh; }
        else { s.sel_need[b] = need - (int)above; s.sel_sh[b] = sh - 8; }
    }
    return done ? 0 : 1;
}

// grid-wide step with rollback on, by ALL threads after sel_grid (sel_need is final): the problems taking a top-K step with a
// clear conflict bit are snapshotted (rb_snap = 1; every other problem gets 0).  A barrier must follow before their fixes.
__device__ __forceinline__ bool rb_takes(const pdp_state& s, int b) {
    return s.sel_need[b] == 0 && !(s.flags[b] & PDP_FLAG_UP_CONFLICT);
}
__device__ __forceinline__ void rb_snapshot_grid(const KArgs& A) {
    const pdp_graph& g = A.g; const pdp_state& s = A.s;
    WARP_STRIDED(b, g.B) {
        if (b >= g.B) continue;
        const bool t = rb_takes(s, (int)b);
        s.rb_snap[b] = t ? 1 : 0;
        if (t) A.rb.is_sat[b] = s.is_sat[b];
    }
    if (range_scans(g)) {   // few contiguous problems: their node ranges
        for (int b = 0; b < (int)g.B; ++b) {
            if (!rb_takes(s, b)) continue;
            for (int i = g.prob_vptr[b] + (int)gtid(); i < g.prob_vptr[b + 1]; i += (int)gthreads()) rb_save_var(A, i);
            for (int a = g.prob_fptr[b] + (int)gtid(); a < g.prob_fptr[b + 1]; a += (int)gthreads()) rb_save_clause(A, a);
        }
        return;
    }
    WARP_STRIDED(i, g.V) { if (i < g.V && rb_takes(s, g.bvm[i])) rb_save_var(A, (int)i); }
    WARP_STRIDED(a, g.F) { if (a < g.F && rb_takes(s, g.bfm[a])) rb_save_clause(A, (int)a); }
}
// by ALL threads after the closure when CTRL_RB is set: the problems rb_mark flagged (rb_snap == 2) go back to the snapshot
__device__ __forceinline__ void rb_restore_grid(const KArgs& A, int iter) {
    const pdp_graph& g = A.g; const pdp_state& s = A.s;
    WARP_STRIDED(b, g.B) { if (b < g.B && s.rb_snap[b] == 2) rb_commit(A, (int)b, iter); }
    if (range_scans(g)) {
        for (int b = 0; b < (int)g.B; ++b) {
            if (s.rb_snap[b] != 2) continue;
            for (int i = g.prob_vptr[b] + (int)gtid(); i < g.prob_vptr[b + 1]; i += (int)gthreads()) rb_restore_var(A, i);
            for (int a = g.prob_fptr[b] + (int)gtid(); a < g.prob_fptr[b + 1]; a += (int)gthreads()) rb_restore_clause(A, a);
        }
        return;
    }
    WARP_STRIDED(i, g.V) { if (i < g.V && s.rb_snap[g.bvm[i]] == 2) rb_restore_var(A, (int)i); }
    WARP_STRIDED(a, g.F) { if (a < g.F && s.rb_snap[g.bfm[a]] == 2) rb_restore_clause(A, (int)a); }
}

// Grid-wide selection over the problems the arg-max phase left selectable (conv, no NaN coefficient, max c > 0); called by
// ALL threads after that phase and a barrier, returns after a barrier.  Problems with K_b >= 2 get arg_idx cleared (the
// arg-max fix skips them) and their final rule in sel_need / sel_sh / sel_pref; every other problem gets sel_need = -1.
// One histogram pass over the variables, then up to 7 more while some problem is undecided (CTRL_SEL parity slots).
template <typename CF>
__device__ __forceinline__ void sel_grid(const KArgs& A, cg::grid_group& grid, const CF& coef, float frac, bool halve) {
    const pdp_graph& g = A.g; const pdp_state& s = A.s;
    for (int pass = 0; pass < 8; ++pass) {
        if (pass > 0 && !s.ctrl[CTRL_SEL + (pass & 1)]) break;   // uniform: written before the last barrier
        const bool first = pass == 0;
        for (int64_t base = gwarp() * 32; base < g.V; base += gwarps() * 32) {
            const int64_t i = base + lane_id();
            int b = 0; bool valid = false;
            if (i < g.V) {
                b = g.bvm[i];
                valid = first ? (s.conv[b] && !s.c_nan[b] && u2f(s.c_max[b]) > 0.f) : (s.sel_need[b] > 0);
            }
            const float c = valid ? coef(i) : 0.f;
            sel_hist_var(s, valid, b, i, c, valid && s.av[i], first);
        }
        if (gtid() == 0) s.ctrl[CTRL_SEL + ((pass + 1) & 1)] = 0;
        grid.sync();
        for (int64_t b = gwarp(); b < g.B; b += gwarps()) {
            int st = -1;
            if (first) {
                if (s.conv[b] && !s.c_nan[b] && u2f(s.c_max[b]) > 0.f) {
                    st = sel_decide(s, (int)b, frac, true, halve);
                    if (st >= 0 && lane_id() == 0) s.arg_idx[b] = 0x7fffffff;
                } else if (lane_id() == 0) {
                    s.sel_need[b] = -1;
                }
            } else if (s.sel_need[b] > 0) {
                st = sel_decide(s, (int)b, frac, false, halve);
            }
            if (st > 0 && lane_id() == 0) s.ctrl[CTRL_SEL + ((pass + 1) & 1)] = 1;
        }
        grid.sync();
    }
}

// ------------------------------------------------------------------------------------------------
// CTA-local decimation.  Everything the decimator does to a converged problem -- scoring, arg-max, fixing
// the variable, unit propagation and pure-literal peeling to closure, the CNF check and the termination
// decision -- touches that problem only, so for problems that one CTA can walk (the common case: thousands of
// n ~ 100 problems per batch) a CTA does all of it with block barriers, where the grid-wide phases above need a
// few dozen grid barriers per iteration.  Same arithmetic and the same synchronous rounds as the grid-wide
// phases (which stay for large problems and batch replication).
// One body, loc_decimate, runs on a view of the problem (local indices i in [0, n), a in [0, m)): LocGlobal works in place
// on the state in global memory, TinyView on a copy staged in shared memory.  A view holds the node arrays and provides the
// clause and variable tests, the fixes, de-activations and scores, and the conflict rollback's save (before a top-K fix),
// restore (after a step that conflicted) and write_back (after any other step).
// ------------------------------------------------------------------------------------------------
struct LocSmem {
    uint32_t cmax, cmin, cnan;
    int arg, flag, conflicts, nunsat, fixed;
};

// what both views hold: problem b (nodes [v0, v0 + n), [f0, f0 + m)), the surveys eta[w], and the node arrays
struct LocNodes {
    const KArgs& A;
    int b, v0, f0, n, m, w;
    float pi;
    uint8_t *av, *af, *pure, *single;
    float *sol, *score;
    int *cnt, *ev;      // unit clauses pointing at the variable, signed sum of those
};

// the problem in place: slices of the state, the global CSR / CSC; de-activations set the edge-mask bits
struct LocGlobal : LocNodes {
    __device__ __forceinline__ float score_of(int i) const { return score_variable(A.g, A.s, A.s.eta[w], v0 + i, pi); }
    __device__ __forceinline__ bool is_unit(int a, int& j, bool& neg) const {
        const bool u = clause_unit(A.g.c_var, A.g.cl_ptr[f0 + a], A.g.cl_ptr[f0 + a + 1], A.s.av, j, neg);
        j -= v0;
        return u;
    }
    __device__ __forceinline__ bool is_pure(int i, float& val) const { return var_pure(A.g, A.s.af, v0 + i, val); }
    __device__ __forceinline__ bool satisfied(int a) const {
        return clause_satisfied(A.g.c_var, A.g.cl_ptr[f0 + a], A.g.cl_ptr[f0 + a + 1], A.s.sol);
    }
    __device__ __forceinline__ void fix(int i, float sg) const { fix_variable(A.g, A.s, v0 + i, sg); }
    __device__ __forceinline__ void drop_clause(int a) const { deactivate_clause(A.g, A.s, f0 + a); }
    __device__ __forceinline__ void drop_var(int i) const { deactivate_variable(A.g, A.s, v0 + i); }
    __device__ __forceinline__ void save(int tid, int nthr) const {
        for (int i = tid; i < n; i += nthr) rb_save_var(A, v0 + i);
        for (int a = tid; a < m; a += nthr) rb_save_clause(A, f0 + a);
    }
    __device__ __forceinline__ void restore(int tid, int nthr) const {
        for (int a = tid; a < m; a += nthr) rb_restore_clause(A, f0 + a);
        for (int i = tid; i < n; i += nthr) rb_restore_var(A, v0 + i);
    }
    __device__ __forceinline__ void write_back(int, int) const {}
};
__device__ __forceinline__ LocGlobal loc_global(const KArgs& A, int b, int w, float pi) {
    const pdp_graph& g = A.g; const pdp_state& s = A.s;
    const int v0 = g.prob_vptr[b], f0 = g.prob_fptr[b];
    return LocGlobal{{A, b, v0, f0, g.prob_vptr[b + 1] - v0, g.prob_fptr[b + 1] - f0, w, pi, s.av + v0, s.af + f0, s.pure + v0,
                      s.single + f0, s.sol + v0, s.score + v0, s.up_cnt + v0, s.up_ev + v0}};
}

// ------------------------------------------------------------------------------------------------
// shared-memory tier of the CTA-local decimation.  A problem whose masks, adjacency (16-bit local indices) and
// scratch fit the group's share of the (idle) sweep buffer is decimated entirely in shared memory: the closure
// is a chain of dozens of dependent rounds, each a couple of microseconds through global memory and tens of
// nanoseconds here.  Global memory keeps the problem as it was until the write-back at the end.
// ------------------------------------------------------------------------------------------------
struct TinyView : LocNodes {
    uint16_t *clp, *cvar, *vp, *vcls;   // local CSR / CSC: pointers, (local index | sign << 15)
    const float* eta_s;                 // the problem's surveys in variable-major order (null: not staged)
    __device__ __forceinline__ float score_of(int i) const {
        if (!eta_s) return score_variable(A.g, A.s, A.s.eta[w], v0 + i, pi);
        float ps = 0.f, ns = 0.f, as = 0.f;   // score_variable on the staged copies (same order, same operations)
        for (int p = vp[i]; p < vp[i + 1]; ++p) {
            const uint32_t cw = vcls[p];
            const float f = L10(1.f - eta_s[p]) * (float)af[cw & 0x7fffu];
            const bool neg = (cw & 0x8000u) != 0u;
            ps += (neg ? 0.f : 1.f) * f;
            ns += (neg ? 1.f : 0.f) * f;
            as += f;
        }
        return sp_score_tail(ps, ns, as, 0.f, 0.f);
    }
    __device__ __forceinline__ bool is_unit(int a, int& j, bool& neg) const { return clause_unit(cvar, clp[a], clp[a + 1], av, j, neg); }
    __device__ __forceinline__ bool is_pure(int i, float& val) const {
        int deg = 0, sdeg = 0;
        for (int p = vp[i]; p < vp[i + 1]; ++p) {
            const uint32_t cw = vcls[p];
            if (af[cw & 0x7fffu]) { ++deg; sdeg += (cw & 0x8000u) ? -1 : 1; }
        }
        val = ((sdeg > 0 ? 1.f : (sdeg < 0 ? -1.f : 0.f)) + 1.f) / 2.0f;
        return deg == abs(sdeg);
    }
    __device__ __forceinline__ bool satisfied(int a) const { return clause_satisfied(cvar, clp[a], clp[a + 1], sol); }
    __device__ __forceinline__ void fix(int i, float sg) const {
        for (int p = vp[i]; p < vp[i + 1]; ++p) {
            const uint32_t w = vcls[p];
            const float lit = (w & 0x8000u) ? -1.f : 1.f;
            if (lit * sg > 0.f) af[w & 0x7fffu] = 0;
        }
        av[i] = 0;
        sol[i] = (sg + 1.f) / 2.0f;
    }
    __device__ __forceinline__ void drop_clause(int a) const { af[a] = 0; }
    __device__ __forceinline__ void drop_var(int i) const { av[i] = 0; }
    __device__ __forceinline__ void save(int, int) const {}
    // the step wrote nothing to global memory: the solution before it is still there
    __device__ __forceinline__ void restore(int tid, int nthr) const {
        for (int i = tid; i < n; i += nthr) sol[i] = A.s.sol[v0 + i];
    }
    // what changed: masks (+ edge-mask bits), solutions
    __device__ __forceinline__ void write_back(int tid, int nthr) const {
        const pdp_graph& g = A.g; const pdp_state& s = A.s;
        for (int i = tid; i < n; i += nthr) {
            if (!av[i] && s.av[v0 + i]) deactivate_variable(g, s, v0 + i);
            s.sol[v0 + i] = sol[i];
        }
        for (int a = tid; a < m; a += nthr)
            if (!af[a] && s.af[f0 + a]) deactivate_clause(g, s, f0 + a);
    }
};
__device__ __forceinline__ size_t tiny_bytes(int n, int m, int E) {
    return (size_t)n * (1 + 1 + 4 + 4 + 4 + 4) + (size_t)m * 2 + (size_t)(m + 1 + n + 1 + 2 * E) * 2 + 64;
}
// problem b staged by its group into `area` (share bytes, at least tiny_bytes of the problem); a barrier must follow
__device__ __forceinline__ TinyView tiny_stage(const KArgs& A, int b, int w, float pi, unsigned char* area, int share, int tid, int nthr) {
    const pdp_graph& g = A.g; const pdp_state& s = A.s;
    const int v0 = g.prob_vptr[b], v1 = g.prob_vptr[b + 1], f0 = g.prob_fptr[b], f1 = g.prob_fptr[b + 1];
    const int n = v1 - v0, m = f1 - f0;
    const int ec0 = g.cl_ptr[f0], ep0 = g.var_ptr[v0], E = g.cl_ptr[f1] - ec0;
    TinyView t{{A, b, v0, f0, n, m, w, pi}};
    float* f = reinterpret_cast<float*>(area);
    t.sol = f; t.score = f + n;
    t.cnt = reinterpret_cast<int*>(f + 2 * n); t.ev = t.cnt + n;
    uint16_t* h = reinterpret_cast<uint16_t*>(t.ev + n);
    t.clp = h; t.vp = t.clp + (m + 1); t.cvar = t.vp + (n + 1); t.vcls = t.cvar + E;
    uint8_t* q = reinterpret_cast<uint8_t*>(t.vcls + E);
    t.av = q; t.pure = q + n; t.af = q + 2 * n; t.single = t.af + m;
    // the surveys of the problem in variable-major order, when they fit too (pi == 0: the external force column drops out)
    const size_t eta_off = (tiny_bytes(n, m, E) + 15) & ~(size_t)15;
    if ((pi == 0.f) && (eta_off + (size_t)E * 4 <= (size_t)share)) {
        float* eta_s = reinterpret_cast<float*>(area + eta_off);
        const float* __restrict__ eta = s.eta[w];
        for (int e = tid; e < E; e += nthr) eta_s[e] = eta[g.p_vpos[ep0 + e]];
        t.eta_s = eta_s;
    }
    for (int i = tid; i < n; i += nthr) {
        t.av[i] = s.av[v0 + i]; t.pure[i] = 0; t.sol[i] = s.sol[v0 + i]; t.cnt[i] = 0; t.ev[i] = 0;
    }
    for (int i = tid; i <= n; i += nthr) t.vp[i] = (uint16_t)(g.var_ptr[v0 + i] - ep0);
    for (int a = tid; a < m; a += nthr) { t.af[a] = s.af[f0 + a]; t.single[a] = 0; }
    for (int a = tid; a <= m; a += nthr) t.clp[a] = (uint16_t)(g.cl_ptr[f0 + a] - ec0);
    for (int e = tid; e < E; e += nthr) {
        const uint32_t cw = g.c_var[ec0 + e];
        t.cvar[e] = (uint16_t)(((cw & PDP_IDX_MASK) - v0) | ((cw & PDP_SIGN_BIT) ? 0x8000u : 0u));
        t.vcls[e] = (uint16_t)((g.v_cls[ep0 + e] - f0) | ((g.v_cedge[ep0 + e] & PDP_SIGN_BIT) ? 0x8000u : 0u));
    }
    return t;
}

#define LSYNC() bar_sync(bar_id, nthr)
// the fractional selection of one converged problem inside its CTA group (sel_grid's passes over the problem's own
// variables, group barriers instead of grid barriers; the histograms stay in global memory: the kernel's shared memory is
// the sweep buffer's).  Called by the whole group after the scoring loop with !cnan and max c > 0.  Returns false for
// K_b == 1 (the caller applies the arg-max rule); otherwise fixes the taken variables and sets ls.fixed (2: with rollback
// on, the view has saved the state before the fix, and the snapshot holds is_sat).
template <typename View>
__device__ __forceinline__ bool loc_select_fix(const View& V, int iter, LocSmem& ls, int tid, int nthr, int bar_id) {
    const KArgs& A = V.A; const pdp_state& s = A.s;
    const int b = V.b;
    for (int pass = 0; pass < 8; ++pass) {
        const bool first = pass == 0;
        if (!first && s.sel_need[b] <= 0) break;
        for (int base = 0; base < V.n; base += nthr) {   // (nthr is a multiple of 32: whole warps take part)
            const int i = base + tid;
            const bool valid = i < V.n;
            const float c = valid ? fabsf(V.score[i]) * (float)V.av[i] : 0.f;
            sel_hist_var(s, valid, b, V.v0 + i, c, valid && V.av[i], first);
        }
        LSYNC();
        if (tid < 32) sel_decide(s, b, A.dec_fraction, first, A.rb.av != nullptr);
        LSYNC();
        if (first && s.sel_need[b] < 0) return false;
    }
    const bool snap = A.rb.av != nullptr && !(s.flags[b] & PDP_FLAG_UP_CONFLICT);
    if (snap) {
        V.save(tid, nthr);
        if (tid == 0) A.rb.is_sat[b] = s.is_sat[b];
        LSYNC();
    }
    bool any = false;
    for (int i = tid; i < V.n; i += nthr) {
        const float c = fabsf(V.score[i]) * (float)V.av[i];
        if (!sel_taken(s, b, V.v0 + i, c, V.av[i] != 0)) continue;
        const float sg = sgnf(V.score[i]);
        V.fix(i, sg);
        any = true;
        record_fix(A, iter, V.v0 + i, sg);
    }
    if (any) { ls.fixed = snap ? 2 : 1; s.masked[b] = 1; s.dirty[b] = 1; }
    LSYNC();
    if (tid == 0) s.sel_need[b] = -1;
    return true;
}

template <typename View>
__device__ __forceinline__ void loc_closure(const View& V, LocSmem& ls, int tid, int nthr, int bar_id) {
    const pdp_state& s = V.A.s;
    const int b = V.b;
    for (;;) {   // unit propagation rounds, solver.py:234-273
        if (tid == 0) { ls.flag = 0; ls.conflicts = 0; }
        LSYNC();
        for (int a = tid; a < V.m; a += nthr) {
            int j; bool neg;
            if (!V.af[a] || !V.is_unit(a, j, neg)) continue;
            V.single[a] = 1;
            atomicAdd(&V.cnt[j], 1);
            atomicAdd(&V.ev[j], neg ? -1 : 1);
            ls.flag = 1;
        }
        LSYNC();
        if (!ls.flag) break;
        for (int i = tid; i < V.n; i += nthr) {
            const int cnt = V.cnt[i];
            if (cnt > 0 && abs(V.ev[i]) != cnt) atomicAdd(&ls.conflicts, 1);
        }
        LSYNC();
        const int nc = ls.conflicts;   // the `== 1` quirk of solver.py:257,261
        for (int a = tid; a < V.m; a += nthr) {
            if (V.single[a]) { V.drop_clause(a); V.single[a] = 0; }
            else if (V.af[a] && nc == 1) V.drop_clause(a);
        }
        for (int i = tid; i < V.n; i += nthr)
            if (V.av[i] && nc == 1) V.drop_var(i);
        if (tid == 0) { s.masked[b] = 1; if (nc >= 1) { s.is_sat[b] = 0.f; s.flags[b] |= PDP_FLAG_UP_CONFLICT; } }
        LSYNC();
        for (int i = tid; i < V.n; i += nthr) {
            const int cnt = V.cnt[i];
            if (cnt > 0) {
                const int ev = V.ev[i];
                V.cnt[i] = 0; V.ev[i] = 0;
                if (V.av[i] && abs(ev) == cnt) V.fix(i, ev > 0 ? 1.f : -1.f);
            }
        }
        LSYNC();
    }
    for (;;) {   // pure-literal peeling rounds, solver.py:188-203
        LSYNC();
        if (tid == 0) ls.flag = 0;
        LSYNC();
        for (int i = tid; i < V.n; i += nthr) {
            float val;
            if (!V.av[i] || !V.is_pure(i, val)) continue;
            V.pure[i] = 1;
            V.sol[i] = val;
            ls.flag = 1;
        }
        LSYNC();
        if (!ls.flag) break;
        // a pure variable is fixed to the value the round gave it: every active clause holding it is satisfied
        // (none holds it: sol 0.5, sign 0, and it only leaves the problem)
        for (int i = tid; i < V.n; i += nthr) {
            if (!V.pure[i]) continue;
            V.pure[i] = 0;
            V.fix(i, 2.f * V.sol[i] - 1.f);
        }
        if (tid == 0) s.masked[b] = 1;
    }
}

// one converged problem: pdp_decimate.py:152-171 + solver.py:275-285 + trainer.py:150-162
template <bool FRAC, typename View>
__device__ __forceinline__ void loc_decimate(const View& V, int iter, bool check_termination, LocSmem& ls, int tid, int nthr, int bar_id) {
    const KArgs& A = V.A; const pdp_state& s = A.s;
    const int b = V.b;
    if (tid == 0) { ls.cmax = 0u; ls.cmin = 0x7f800000u; ls.cnan = 0u; ls.arg = 0x7fffffff; ls.fixed = 0; ls.nunsat = 0; }
    LSYNC();
    for (int i = tid; i < V.n; i += nthr) {
        const float sc = V.score_of(i);
        V.score[i] = sc;
        const float c = fabsf(sc) * (float)V.av[i];
        if (c != c) ls.cnan = 1u; else { atomicMax(&ls.cmax, f2u(c)); atomicMin(&ls.cmin, f2u(c)); }
    }
    LSYNC();
    const bool topk = FRAC && !ls.cnan && u2f(ls.cmax) > 0.f && loc_select_fix(V, iter, ls, tid, nthr, bar_id);
    if (!topk && !ls.cnan) {   // first index attaining max of fl(fl(c - min) + 1), util.py:257-265
        const float mn = u2f(ls.cmin);
        const float kmax = argmax_key(u2f(ls.cmax), mn);
        for (int i = tid; i < V.n; i += nthr) {
            const float c = fabsf(V.score[i]) * (float)V.av[i];
            if (argmax_key(c, mn) == kmax) atomicMin(&ls.arg, i);
        }
    }
    LSYNC();
    if (!topk && tid == 0 && !ls.cnan && u2f(ls.cmax) > 0.f && ls.arg != 0x7fffffff) {
        const int i = ls.arg;
        const float sg = sgnf(V.score[i]);
        if (sg != 0.f && V.av[i]) {
            V.fix(i, sg);
            s.masked[b] = 1; s.dirty[b] = 1;
            ls.fixed = 1;
            record_fix(A, iter, V.v0 + i, sg);
        }
    }
    LSYNC();
    if (ls.fixed) {
        loc_closure(V, ls, tid, nthr, bar_id);
        if (FRAC && ls.fixed == 2 && (s.flags[b] & PDP_FLAG_UP_CONFLICT)) {   // conflict rollback
            V.restore(tid, nthr);
            LSYNC();   // everybody has read the conflict bit before it is cleared
            if (tid == 0) rb_commit(A, b, iter);
        } else {
            V.write_back(tid, nthr);
        }
    }
    LSYNC();
    if (s.dirty[b]) {
        if (check_termination) {   // SatCNFEvaluator on _solution over the full formula, then trainer.py:150-162
            int nun = 0;
            for (int a = tid; a < V.m; a += nthr) nun += V.satisfied(a) ? 0 : 1;
            nun = __reduce_add_sync(0xffffffffu, nun);
            if ((tid & 31) == 0 && nun) atomicAdd(&ls.nunsat, nun);
            LSYNC();
            if (tid == 0) {
                if (ls.nunsat == 0) {
                    if (s.active[b]) { s.active[b] = 0; s.freeze_iter[b] = iter; atomicSub(&s.ctrl[CTRL_NUM_ACTIVE], 1); }
                    s.flags[b] |= PDP_FLAG_SOLVED;
                }
                s.dirty[b] = 0; s.n_unsat[b] = 0;
            }
        } else if (tid == 0) {
            s.ctrl[CTRL_ANY_DIRTY] = 1;
        }
    }
    if (tid == 0) s.conv[b] = 0;
    LSYNC();
}
#undef LSYNC

__device__ __forceinline__ bool loc_problem_is_small(const pdp_graph& g, int b) {
    return (g.prob_vptr[b + 1] - g.prob_vptr[b] <= PDP_LOCAL_MAX_V) && (g.prob_fptr[b + 1] - g.prob_fptr[b] <= PDP_LOCAL_MAX_F);
}

// groups of PDP_LOCAL_GROUP threads (named barriers 8..15) take one problem each
#define PDP_LOCAL_GROUP 128
// `area` / `area_bytes`: the CTA's dynamic shared memory (the sweep buffer, idle during the decimation), split evenly
// between the groups; null when the kernel has none
// (one array for both instances of loc_decimate_all)
__device__ __forceinline__ LocSmem* loc_smem() {
    __shared__ LocSmem ls[8];
    return ls;
}
template <bool FRAC>
__device__ __forceinline__ void loc_decimate_all(const KArgs& A, int iter, int w, float pi, bool check_termination,
                                                 unsigned char* area, int area_bytes) {
    LocSmem* ls = loc_smem();
    const pdp_state& s = A.s;
    int ngroups = blockDim.x / PDP_LOCAL_GROUP;
    if (ngroups > 8) ngroups = 8;
    const int gthr = blockDim.x / ngroups;           // threads per group (a multiple of 32)
    const int grp = threadIdx.x / gthr, gt = threadIdx.x % gthr;
    // the groups drain the queue decide_phase filled (the order is irrelevant: problems do not interact)
    const int count = s.ctrl[CTRL_LOC_COUNT];
    for (;;) {
        if (gt == 0) ls[grp].flag = atomicAdd(&s.ctrl[CTRL_LOC_NEXT], 1);
        bar_sync(8 + grp, gthr);
        const int k = ls[grp].flag;
        bar_sync(8 + grp, gthr);
        if (k >= count) break;
        const int b = s.loc_list[k];
        const int share = area ? ((area_bytes / ngroups) & ~15) : 0;
        const int n = A.g.prob_vptr[b + 1] - A.g.prob_vptr[b], m = A.g.prob_fptr[b + 1] - A.g.prob_fptr[b];
        const int E = A.g.cl_ptr[A.g.prob_fptr[b + 1]] - A.g.cl_ptr[A.g.prob_fptr[b]];
        if (n < 32768 && m < 32768 && E < 65536 && tiny_bytes(n, m, E) <= (size_t)share)
            loc_decimate<FRAC>(tiny_stage(A, b, w, pi, area + (size_t)grp * share, share, gt, gthr), iter, check_termination,
                               ls[grp], gt, gthr, 8 + grp);
        else
            loc_decimate<FRAC>(loc_global(A, b, w, pi), iter, check_termination, ls[grp], gt, gthr, 8 + grp);
    }
}

// ------------------------------------------------------------------------------------------------
// full-formula satisfaction count (SatCNFEvaluator on _solution, util.py:210-236) for dirty problems
// ------------------------------------------------------------------------------------------------
__device__ __forceinline__ void cnf_count_dirty(const KArgs& A) {
    const pdp_graph& g = A.g; const pdp_state& s = A.s;
    KeyedReducer<CountAcc> red;
    const bool native = s.ctrl[CTRL_NATIVE] != 0;
    if (range_scans(g)) {
        for (int b = 0; b < (int)g.B; ++b) {
            if (!s.dirty[b]) continue;
            const int f1 = g.prob_fptr[b + 1];
            red.touch(s, b);
            for (int a = g.prob_fptr[b] + (int)gtid(); a < f1; a += (int)gthreads()) {
                if (native && s.af[a]) { red.acc.n += 1; continue; }
                red.acc.n += clause_satisfied(g.c_var, g.cl_ptr[a], g.cl_ptr[a + 1], s.sol) ? 0 : 1;
            }
            red.finish(s);
        }
        return;
    }
    WARP_STRIDED(a, g.F) {
        if (a >= g.F) continue;
        const int b = g.bfm[a];
        if (!s.dirty[b]) continue;
        red.touch(s, b);
        if (native && s.af[a]) { red.acc.n += 1; continue; }   // an active clause holds no true literal (CTRL_NATIVE)
        red.acc.n += clause_satisfied(g.c_var, g.cl_ptr[a], g.cl_ptr[a + 1], s.sol) ? 0 : 1;
    }
    red.finish(s);
}
