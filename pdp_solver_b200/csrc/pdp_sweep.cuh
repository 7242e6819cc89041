// pdp_sweep.cuh -- the blocked shared-memory passes of the SP sweep (product path of pdp_sp_run, included by
// pdp_device.cuh).  Layout: pdp_common.cuh / DESIGN.md.  One CTA walks blocks of whole nodes; per block
//     load      the block's message region comes into shared memory AS IT LIES in global memory, by bulk-asynchronous
//               copies (cp.async.bulk.shared.global + mbarrier complete_tx: issued by one thread, no registers, no issue
//               slots; the other CTA of the SM computes meanwhile).  The run table of the write-out and the run offsets
//               ride along;
//     node      the per-node arithmetic IN PLACE: a 16-bit table (g.cfwd / g.vfwd), read once per pass and coalesced in node
//               order, gives the region position x of every node-order slot; the node reads plane[x] and puts its result
//               back into plane[x].
//                 clauses: a thread owns a clause, its K table entries are consecutive;
//                 variables: a WARP owns 32 variables of (nearly) equal degree and the table stores their entries
//                 transposed -- row j of the group holds the j-th edge of every member that has one, lane l reads entry
//                 `row start + l`; the ascending-edge accumulation order of the reference (torch.mm(sparse, dense) on
//                 CPU) is the row order;
//     write-out the plane streams out in region order = ascending destination order.  Consecutive slots hit consecutive
//               destinations (a RUN: the edges between this block and one block of the other side), so destinations are
//               not stored per edge: one bit per slot marks the start of a run, one 32-bit count per 32 slots gives the
//               run index, one 32-bit offset per run gives `destination - slot`.  No global load in this phase.
// A slot's value in the plane carries two markers for the write-out (results are >= +0 or NaN):
//     PDP_SLOT_SKIP (-inf)   the node left the slot alone (frozen problem inside a block that still has work);
//     sign bit               the problem is on the sticky-NaN path: keep a NaN that is already stored at the destination
//                            (the reference blends mask*new + (1-mask)*old arithmetically: 0*NaN = NaN, pdp_propagate.py:175,218).
// Dynamic shared memory of a CTA (SweepCfg<CTAS>::kSmem bytes):
//   [0, kPlaneBytes)       clause pass: plane X;  variable pass: planes PA | PB (kPlaneV words each)
//   then 8 * kRunWords     run table words of the block
//   then 4 * kAdjCap       run offsets of the block
#pragma once

#define PDP_SLOT_SKIP 0xff800000u

__device__ __forceinline__ bool blk_problem_runs(const pdp_state& s, int b) { return s.active[b] != 0; }

// true when no problem in [b0, b1] is to be processed by the blocked passes (uniform over the CTA)
__device__ __forceinline__ bool blk_idle(const pdp_state& s, int b0, int b1) {
    if (b0 == b1) return !blk_problem_runs(s, b0);
    int any = 0;
    for (int b = b0 + (int)threadIdx.x; b <= b1; b += (int)blockDim.x) any |= blk_problem_runs(s, b) ? 1 : 0;
    return __syncthreads_or(any) == 0;
}

#ifndef PDP_UNROLL_WO
#define PDP_UNROLL_WO 4    // write-out: slots per thread in flight
#endif
#ifndef PDP_COLD
#define PDP_COLD __forceinline__
#endif

// ------------------------------------------------------------------------------------------------
// bulk-asynchronous copies global -> shared (the 1-D form of TMA) completing on an mbarrier
// ------------------------------------------------------------------------------------------------
__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }
__device__ __forceinline__ void mbar_init(uint64_t* bar, int count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count) : "memory");
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
}
__device__ __forceinline__ void mbar_expect_tx(uint64_t* bar, uint32_t bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}
// dst, src 16-byte aligned, bytes a multiple of 16
__device__ __forceinline__ void bulk_g2s(void* dst, const void* src, uint32_t bytes, uint64_t* bar) {
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];"
                 ::"r"(smem_u32(dst)), "l"(src), "r"(bytes), "r"(smem_u32(bar)) : "memory");
}
// generic-proxy accesses of this thread (and, after a barrier, of the CTA) ordered before later async-proxy accesses
__device__ __forceinline__ void fence_proxy_async() { asm volatile("fence.proxy.async;" ::: "memory"); }
// ... the same for shared memory only (before a bulk copy overwrites a plane the CTA has just read): does not wait for the
// thread's outstanding global stores, which the full fence does (3 000 cycles per block right after a write-out, measured)
__device__ __forceinline__ void fence_proxy_async_smem() { asm volatile("fence.proxy.async.shared::cta;" ::: "memory"); }
// one thread: [p, p + bytes) -> L2, rounded outwards to 16-byte units (a hint: no completion to wait for)
__device__ __forceinline__ void bulk_prefetch_l2(const void* p, int bytes) {
    if (bytes <= 0) return;
    const uintptr_t a = (uintptr_t)p & ~(uintptr_t)15;
    const uint32_t n = (uint32_t)((((uintptr_t)p + bytes + 15) & ~(uintptr_t)15) - a);
    asm volatile("cp.async.bulk.prefetch.L2.global [%0], %1;" ::"l"(a), "r"(n) : "memory");
}
// all threads: wait for the phase with this parity.  A copy that never completes (a bug) traps instead of hanging the device.
__device__ __forceinline__ void mbar_wait(uint64_t* bar, uint32_t parity) {
    const uint32_t a = smem_u32(bar);
    uint32_t done = 0;
    long long t0 = 0;
    for (int spin = 0; !done; ++spin) {
        asm volatile("{\n\t.reg .pred p;\n\tmbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\tselp.u32 %0, 1, 0, p;\n\t}"
                     : "=r"(done) : "r"(a), "r"(parity) : "memory");
        if (!done && spin > 64) {
            if (t0 == 0) t0 = clock64();
            else if (clock64() - t0 > (1ll << 32)) __trap();
        }
    }
}

// the whole CTA waits for a phase: one warp polls the barrier word, the others sleep at the block barrier (a polling warp
// takes issue slots from the SM's other CTA: 512 polling threads were 4.5 % of the kernel's instructions).  The polling
// warp's acquire and the block barrier order the copied bytes before every thread's reads.
__device__ __forceinline__ void mbar_wait_cta(uint64_t* bar, uint32_t parity) {
    if (threadIdx.x < 32) mbar_wait(bar, parity);
    __syncthreads();
}

// explicit shared-window accesses (32-bit addresses).  The node phases index the planes through the position table; as
// volatile statements these keep the order they are written in, which is how two rows are interleaved by hand below.
__device__ __forceinline__ uint32_t lds_u32(uint32_t a) { uint32_t v; asm volatile("ld.shared.u32 %0, [%1];" : "=r"(v) : "r"(a)); return v; }
__device__ __forceinline__ float lds_f32(uint32_t a) { float v; asm volatile("ld.shared.f32 %0, [%1];" : "=f"(v) : "r"(a)); return v; }
__device__ __forceinline__ void sts_f32(uint32_t a, float v) { asm volatile("st.shared.f32 [%0], %1;" ::"r"(a), "f"(v)); }
__device__ __forceinline__ void sts_u32(uint32_t a, uint32_t v) { asm volatile("st.shared.u32 [%0], %1;" ::"r"(a), "r"(v)); }

// geometry of one block of a pass: one 48-byte descriptor (three 16-byte loads)
struct BlkGeo {
    int n0, n1;      // node range
    int e0, ne;      // first slot / slots
    int b0, b1;      // problem range
    int run0, nruns; // write-out runs of the block: [run0, run0 + nruns)
    int t0, tn;      // first entry / entries of the block in the position table
    __device__ __forceinline__ bool multi() const { return b0 != b1; }
};
__device__ __forceinline__ BlkGeo load_block(const pdp_blk* __restrict__ desc, int blk) {
    const int4* p = reinterpret_cast<const int4*>(desc + blk);
    const int4 a = __ldg(p), b = __ldg(p + 1), c = __ldg(p + 2);
    BlkGeo B;
    B.n0 = a.x; B.n1 = a.y; B.e0 = a.z; B.ne = a.w; B.b0 = b.x; B.b1 = b.y; B.run0 = b.z; B.nruns = b.w; B.t0 = c.x; B.tn = c.y;
    return B;
}
__device__ __forceinline__ BlkGeo clause_block(const pdp_graph& g, int blk) { return load_block(g.cb_desc, blk); }
__device__ __forceinline__ BlkGeo var_block(const pdp_graph& g, int blk) { return load_block(g.vb_desc, blk); }

// Where the pieces of a block land in shared memory.  Bulk copies move whole 16-byte units: every source range is widened
// to 16-byte boundaries and the consumer indexes with the offset of its first element.
struct BlkStage {
    int a0, nbytes;      // message region: first element copied (a multiple of 4 <= e0), bytes
    int shift;           // e0 - a0: region position x sits at plane[shift + x]
    int w0, wbytes;      // run table: first word copied (even, <= e0 >> 5), bytes
    int r0, rbytes;      // run offsets: first offset copied (a multiple of 4 <= run0), bytes (0: not staged, the write-out reads g.*_wadj)
};
template <int CAP>
__device__ __forceinline__ BlkStage blk_stage(const BlkGeo& B) {
    BlkStage S;
    S.a0 = B.e0 & ~3;
    S.shift = B.e0 - S.a0;
    S.nbytes = 4 * (((B.e0 + B.ne + 3) & ~3) - S.a0);
    S.w0 = (B.e0 >> 5) & ~1;
    S.wbytes = 8 * (((((B.e0 + B.ne - 1) >> 5) + 2) & ~1) - S.w0);
    S.r0 = B.run0 & ~3;
    const int nr = ((B.run0 + B.nruns + 3) & ~3) - S.r0;
    S.rbytes = nr <= CAP ? 4 * nr : 0;
    return S;
}

// write-out: slots [wlo, wend) of the block's region (all of it); destinations ascend.  One slot per thread and
// instruction (with several consecutive slots per thread a warp's stores would be strided and every destination sector
// written several times).  Everything but the store (and the rare sticky re-read) is shared memory, addressed in the shared
// window: plane_sa = address of slot 0's word (slot w at plane_sa + 4 w), wrun_sa = address of run table word 0 (word i at
// wrun_sa + 8 i), adj_sa = address of run 0's offset (ADJ_S) or adj_g = g.*_wadj (a block with too many runs to stage).
// MARK: the block may hold markers (several problems, or a problem on the sticky-NaN path).  Without them a row costs no
// vote and no branch; the sign bit is cleared on the way out (a NaN result may carry one).
template <int G, bool ADJ_S, bool MARK>
__device__ __forceinline__ void ph_write_out_t(int t, int wlo, int wend, uint32_t plane_sa, uint32_t wrun_sa, uint32_t adj_sa,
                                               const int32_t* __restrict__ adj_g, const float* old, float* out) {   // old may alias out (q is updated in place)
    // A warp takes 32 slots that share one word of the run table: slot w = row + lane with row a multiple of 32, so the
    // lane's bit mask is fixed and the table word is one broadcast load.  Rows that lie entirely inside [wlo, wend) go
    // through the main loop without a bounds check; the (at most two) partial rows at the ends are left to two warps.
    const int lane = t & 31, warp = t >> 5;
    uint32_t lmask;
    asm("mov.u32 %0, %%lanemask_le;" : "=r"(lmask));
    auto dest = [&](int w, uint32_t rbx, uint32_t rby) {
        const int run = (int)rby + __popc(rbx & lmask);
        return w + (ADJ_S ? (int)lds_u32(adj_sa + 4u * (uint32_t)run) : __ldg(adj_g + run));
    };
    auto special = [&](int d, uint32_t raw) {       // a slot with a marker (sign bit): skipped, or sticky
        if (raw == PDP_SLOT_SKIP) return;
        raw &= 0x7fffffffu;                         // sticky (or a NaN that happens to carry a sign: harmless)
        const float ov = old[d];
        if (ov != ov) raw = __float_as_uint(ov);
        out[d] = __uint_as_float(raw);
    };
    const int rf0 = (wlo + 31) & ~31, rf1 = wend & ~31;      // full rows: [rf0, rf1)
    constexpr int U = PDP_UNROLL_WO;
    int row = rf0 + 32 * warp;
    uint32_t pa = plane_sa + 4u * (uint32_t)(row + lane), wa = wrun_sa + 8u * (uint32_t)(row >> 5);
    for (; row + (U - 1) * G < rf1; row += U * G, pa += 4u * U * G, wa += 8u * U * (G / 32)) {
        uint32_t raw[U], rbx[U], rby[U];
#pragma unroll
        for (int u = 0; u < U; ++u) {
            raw[u] = lds_u32(pa + 4u * u * G);
            asm volatile("ld.shared.v2.u32 {%0, %1}, [%2];" : "=r"(rbx[u]), "=r"(rby[u]) : "r"(wa + 8u * u * (G / 32)));
        }
#pragma unroll
        for (int u = 0; u < U; ++u) {
            const int d = dest(row + u * G + lane, rbx[u], rby[u]);
            if (!MARK) out[d] = __uint_as_float(raw[u] & 0x7fffffffu);
            else if (!__any_sync(0xffffffffu, (int32_t)raw[u] < 0)) out[d] = __uint_as_float(raw[u]);      // the rule: no marker in the row
            else if ((int32_t)raw[u] < 0) special(d, raw[u]);
            else out[d] = __uint_as_float(raw[u]);
        }
    }
    for (; row < rf1; row += G, pa += 4u * G, wa += 8u * (G / 32)) {
        uint32_t rbx, rby;
        const uint32_t raw = lds_u32(pa);
        asm volatile("ld.shared.v2.u32 {%0, %1}, [%2];" : "=r"(rbx), "=r"(rby) : "r"(wa));
        const int d = dest(row + lane, rbx, rby);
        if (!MARK) out[d] = __uint_as_float(raw & 0x7fffffffu);
        else if ((int32_t)raw < 0) special(d, raw); else out[d] = __uint_as_float(raw);
    }
    // partial rows: the one holding wlo (when wlo is not a multiple of 32) and the one holding wend - 1
    const int r_head = wlo & ~31, r_tail = (wend - 1) & ~31;
    int er = -1;
    if (warp == 0 && r_head < rf0) er = r_head;
    else if (warp == 1 && r_tail >= rf1 && !(r_tail == r_head && r_head < rf0)) er = r_tail;
    if (er >= 0) {
        const int w = er + lane;
        if (w >= wlo && w < wend) {
            uint32_t rbx, rby;
            const uint32_t raw = lds_u32(plane_sa + 4u * (uint32_t)w);
            asm volatile("ld.shared.v2.u32 {%0, %1}, [%2];" : "=r"(rbx), "=r"(rby) : "r"(wrun_sa + 8u * (uint32_t)(er >> 5)));
            const int d = dest(w, rbx, rby);
            if (!MARK) out[d] = __uint_as_float(raw & 0x7fffffffu);
            else if ((int32_t)raw < 0) special(d, raw); else out[d] = __uint_as_float(raw);
        }
    }
}
template <int G>
__device__ __forceinline__ void ph_write_out(int t, const BlkGeo& B, int wlo, int wend, const float* plane, const uint2* wrun_s, int w0,
                                             const int32_t* adj_s, int r0, const int32_t* adj_g, const float* old, float* out, bool marks) {
    const uint32_t plane_sa = smem_u32(plane) - 4u * (uint32_t)B.e0;
    const uint32_t wrun_sa = smem_u32(wrun_s) - 8u * (uint32_t)w0;
    if (adj_s) {
        if (!marks) ph_write_out_t<G, true, false>(t, wlo, wend, plane_sa, wrun_sa, smem_u32(adj_s) - 4u * (uint32_t)r0, adj_g, old, out);
        else ph_write_out_t<G, true, true>(t, wlo, wend, plane_sa, wrun_sa, smem_u32(adj_s) - 4u * (uint32_t)r0, adj_g, old, out);
    } else ph_write_out_t<G, false, true>(t, wlo, wend, plane_sa, wrun_sa, 0u, adj_g, old, out);
}

// the edge-mask bits of the block's region (indexed by layout position) -> sign bits of the plane (its values are >= +0 or
// NaN).  Only the words that have a bit set cost anything.  The first two words of every thread (all of them at the block
// sizes of the two-CTA configuration) are fetched BEFORE the CTA waits for the block's copies: their latency hides there.
struct MaskWords { uint32_t m0, m1; };
template <int G>
__device__ __forceinline__ MaskWords ph_mask_fetch(int t, const uint32_t* __restrict__ mask, const BlkGeo& B) {
    MaskWords M;
    const int W0 = B.e0 >> 5, W1 = (B.e0 + B.ne - 1) >> 5;
    M.m0 = (W0 + t <= W1) ? __ldcg(mask + W0 + t) : 0u;
    M.m1 = (W0 + t + G <= W1) ? __ldcg(mask + W0 + t + G) : 0u;
    return M;
}
template <int G>
__device__ __forceinline__ void ph_apply_mask(int t, const uint32_t* __restrict__ mask, const BlkGeo& B, float* plane, const MaskWords& M) {
    uint32_t* pl = reinterpret_cast<uint32_t*>(plane) - B.e0;
    const int W0 = B.e0 >> 5, W1 = (B.e0 + B.ne - 1) >> 5, wend = B.e0 + B.ne;
    int k = 0;
    for (int i = W0 + t; i <= W1; i += G, ++k) {
        uint32_t m = (k == 0) ? M.m0 : ((k == 1) ? M.m1 : __ldcg(mask + i));
        while (m) {
            const int pos = 32 * i + __ffs(m) - 1;
            m &= m - 1;
            if (pos >= B.e0 && pos < wend) pl[pos] |= 0x80000000u;
        }
    }
}

// one clause of K literals: surveys in place.  X: shifted plane; fw: the clause's K table entries.  MASKED: the sign bit of a
// loaded q marks a masked edge (x = log(q) * 0).  stk: sign bit to put on the results.  Returns whether a NaN was produced.
template <int K, bool MASKED>
__device__ __forceinline__ bool blk_clause_body(float* X, const int (&pos)[K], uint32_t stk) {
    float x[K];
    float tot = 0.f;
#pragma unroll
    for (int j = 0; j < K; ++j) {
        const uint32_t raw = __float_as_uint(X[pos[j]]);
        float v = L40(__uint_as_float(MASKED ? (raw & 0x7fffffffu) : raw));
        if (MASKED && (int32_t)raw < 0) v = v * 0.f;
        x[j] = v;
        tot += v;
    }
    bool made_nan = false;
#pragma unroll
    for (int j = 0; j < K; ++j) {
        const float nv = X30(tot - x[j]);
        made_nan |= (nv != nv);
        X[pos[j]] = __uint_as_float(__float_as_uint(nv) | stk);
    }
    return made_nan;
}
template <bool MASKED>
__device__ __forceinline__ bool blk_clause_body_any(float* X, const uint16_t* __restrict__ fw, int k, uint32_t stk) {
    float tot = 0.f;
    for (int j = 0; j < k; ++j) {
        const uint32_t raw = __float_as_uint(X[fw[j]]);
        float v = L40(__uint_as_float(MASKED ? (raw & 0x7fffffffu) : raw));
        if (MASKED && (int32_t)raw < 0) v = v * 0.f;
        tot += v;
    }
    bool made_nan = false;
    // (a second pass over the inputs: a slot is overwritten right after its own value has been used, the slots differ)
    for (int j = 0; j < k; ++j) {
        const int p = fw[j];
        const uint32_t raw = __float_as_uint(X[p]);
        float v = L40(__uint_as_float(MASKED ? (raw & 0x7fffffffu) : raw));
        if (MASKED && (int32_t)raw < 0) v = v * 0.f;
        const float nv = X30(tot - v);
        made_nan |= (nv != nv);
        X[p] = __uint_as_float(__float_as_uint(nv) | stk);
    }
    return made_nan;
}

// clause pass, node phase: thread per clause.  Blocks whose clauses all have K literals: the table entries of a thread's
// next clause are fetched while the current one is worked on.
template <int G, int K, bool MASKED>
__device__ __forceinline__ void ph_clause_node_k(int t, const pdp_graph& g, const pdp_state& s, const BlkGeo& B, float* X, uint32_t stk_blk) {
    const bool multi = B.multi();
    const uint16_t* __restrict__ fw = g.cfwd + B.t0 + K * t;      // entries of clause n0 + t; the thread's next clause is G further
    int a = B.n0 + t;
    int nxt[K];
#pragma unroll
    for (int j = 0; j < K; ++j) nxt[j] = (a < B.n1) ? (int)fw[j] : 0;
    for (; a < B.n1; a += G) {
        int pos[K];
#pragma unroll
        for (int j = 0; j < K; ++j) pos[j] = nxt[j];
        fw += K * G;
        if (a + G < B.n1) {
#pragma unroll
            for (int j = 0; j < K; ++j) nxt[j] = fw[j];
        }
        int b = B.b0;
        uint32_t stk = stk_blk;
        if (multi) {
            b = g.bfm[a];
            if (!blk_problem_runs(s, b)) {
#pragma unroll
                for (int j = 0; j < K; ++j) X[pos[j]] = __uint_as_float(PDP_SLOT_SKIP);
                continue;
            }
            stk = s.nanflag[b] ? 0x80000000u : 0u;
        }
        if (blk_clause_body<K, MASKED>(X, pos, stk)) s.nanpend[b] = 1;
    }
}
// ... and blocks of mixed clause degrees
template <int G, bool MASKED>
__device__ __forceinline__ void ph_clause_node_any(int t, const pdp_graph& g, const pdp_state& s, const BlkGeo& B, float* X, uint32_t stk_blk) {
    const bool multi = B.multi();
    const uint16_t* __restrict__ fwb = g.cfwd + B.t0;     // entry of clause-major slot c: fwb[c - e0]
    for (int a = B.n0 + t; a < B.n1; a += G) {
        const int lo = g.cl_ptr[a] - B.e0, k = g.cl_ptr[a + 1] - B.e0 - lo;
        const uint16_t* __restrict__ fw = fwb + lo;
        int b = B.b0;
        uint32_t stk = stk_blk;
        if (multi) {
            b = g.bfm[a];
            if (!blk_problem_runs(s, b)) {
                for (int j = 0; j < k; ++j) X[fw[j]] = __uint_as_float(PDP_SLOT_SKIP);
                continue;
            }
            stk = s.nanflag[b] ? 0x80000000u : 0u;
        }
        if (blk_clause_body_any<MASKED>(X, fw, k, stk)) s.nanpend[b] = 1;
    }
}
// ku = common degree of the block's clauses (0: mixed)
template <int G, bool MASKED>
__device__ __forceinline__ void ph_clause_node(int t, const pdp_graph& g, const pdp_state& s, const BlkGeo& B, int ku, float* X, uint32_t stk_blk) {
    switch (ku) {
        case 3: ph_clause_node_k<G, 3, MASKED>(t, g, s, B, X, stk_blk); break;
        case 4: ph_clause_node_k<G, 4, MASKED>(t, g, s, B, X, stk_blk); break;
        case 5: ph_clause_node_k<G, 5, MASKED>(t, g, s, B, X, stk_blk); break;
        case 2: ph_clause_node_k<G, 2, MASKED>(t, g, s, B, X, stk_blk); break;
        default: ph_clause_node_any<G, MASKED>(t, g, s, B, X, stk_blk); break;
    }
}

// statistics of multi-problem blocks: per block-local problem in shared memory
#define PDP_STAT_SLOTS 64
struct BlkStats {
    uint32_t mx0[PDP_STAT_SLOTS], mn0[PDP_STAT_SLOTS], mx1[PDP_STAT_SLOTS], mn1[PDP_STAT_SLOTS], nan[PDP_STAT_SLOTS], nav[PDP_STAT_SLOTS];
};

// branch-free select on a sign mask (all ones / all zeros): one LOP3
__device__ __forceinline__ float fsel(uint32_t mask, float a, float b) {
    return __uint_as_float((__float_as_uint(a) & mask) | (__float_as_uint(b) & ~mask));
}
__device__ __forceinline__ float fand(uint32_t mask, float a) { return __uint_as_float(__float_as_uint(a) & mask); }

// One warp-group of a variable block: 32 variables of consecutive rank in the block's descending-degree order
// (g.vsort), lane l <-> rank 32 * group + l.  The group owns 64 * ceil(degree of its first member / 2) entries of the
// position table from its base (a multiple of 64): rows go in pairs, the 16-bit entries of rows 2k and 2k+1 of lane l sit side
// by side at base + 64 k + 2 l (one 32-bit load per row pair).  Entries of members with fewer edges than the first one are
// padding (never written; read only as the unused half of a pair): 2-7 % of a block.
struct VarGroup {
    int i, deg, base, maxdeg;
    bool have;
};
__device__ __forceinline__ VarGroup var_group(const pdp_graph& g, const BlkGeo& B, int grp) {
    VarGroup V;
    const int ti = B.n0 + grp * 32 + lane_id();
    V.have = ti < B.n1;
    V.i = 0; V.deg = 0; V.base = 0;
    if (V.have) { const int2 ve = __ldg(&g.vsort[ti]); V.i = ve.x; V.base = ve.y & 0xffff; V.deg = (int)((unsigned)ve.y >> 16); }
    V.base = __shfl_sync(0xffffffffu, V.base, 0);     // every entry of a group carries the group's base; lane 0 exists
    V.maxdeg = __shfl_sync(0xffffffffu, V.deg, 0);
    return V;
}
// groups of a block are handed to the warps round by round, odd rounds in reverse (every warp gets high and low degrees)
#define VAR_GROUP_LOOP(grp, B, G, t)                                                                        \
    for (int _gb = 0, _rd = 0, _ng = ((B).n1 - (B).n0 + 31) >> 5, grp; _gb < _ng; _gb += (G) / 32, ++_rd)   \
        if ((grp = (_rd & 1) ? _gb + ((G) / 32 - 1 - ((t) >> 5)) : _gb + ((t) >> 5)) < _ng)

// variable pass, SurveyScorer (pdp_predict.py:155-192) of the variables whose problem asked for it (want_score): same
// operations and order as score_variable() on the new surveys held in PA (sign bit = edge masked; for an active variable
// the edge mask is the clause mask the scorer multiplies with, an inactive variable's score is never looked at) and the
// literal signs of the table.  pi == 0 on the blocked path: the external force does not enter.
// (The reference's pos / neg incidence products hold explicit zeros, 0 * f: they only matter when f is NaN, and then
// the sum over all edges is NaN as well and with it bias and the score: the per-sign sums skip them.)
template <int G>
__device__ __forceinline__ void ph_var_score(int t, const pdp_graph& g, const pdp_state& s, const BlkGeo& B, const float* __restrict__ PA) {
    VAR_GROUP_LOOP(grp, B, G, t) {
        const VarGroup V = var_group(g, B, grp);
        if (!(V.have && s.want_score[B.multi() ? g.bvm[V.i] : B.b0])) continue;
        float ps = 0.f, ns = 0.f, as = 0.f;
        const uint32_t* __restrict__ fw = reinterpret_cast<const uint32_t*>(g.vfwd + B.t0 + V.base) + lane_id();
        for (int j = 0; j < V.deg; ++j) {
            const uint32_t en = (fw[32 * (j >> 1)] >> (16 * (j & 1))) & 0xffffu;
            const uint32_t nb = __float_as_uint(PA[en & 0x7fffu]);
            const uint32_t negm = 0u - (en >> 15);
            const float f = L10(1.f - __uint_as_float(nb & 0x7fffffffu)) * ((nb >> 31) ? 0.f : 1.f);
            ps += fand(~negm, f);
            ns += fand(negm, f);
            as += f;
        }
        s.score[V.i] = sp_score_tail(ps, ns, as, 0.f, 0.f);
    }
}

// variable pass, node phase: ordered sums, decimator statistics, update.  PA: eta(t) (sign bit = edge masked), then q(t);
// PB: eta(t-1), then y.  Both shifted planes, indexed by region position.
// (As in the scorer, the explicit zeros 0 * y of the reference's per-sign sums are skipped: a NaN y makes the sum of its
// own sign NaN, and every message of the variable reads both sums -- `same` the one of its sign, `opp` the other.)
// MULTI: the block holds several problems: frozen ones are left alone (PDP_SLOT_SKIP), those on the sticky-NaN path get
// the sticky sign.
// REINF: reinforce (pdp_set_reinforce) with the external force uniform over each variable's edges: its pi terms are two
// per-variable constants, read from the variable's first edge
template <int G, bool MULTI, bool MASKED, bool PREV, bool REINF>
__device__ __forceinline__ void ph_var_node(int t, const pdp_graph& g, const pdp_state& s, const BlkGeo& B, bool use_mask,
                                            bool em_set, float* __restrict__ PA, float* __restrict__ PB, uint32_t stk_blk,
                                            KeyedReducer<StatAcc>& red, BlkStats& sm_st, bool local_stats, float pi) {
    const int lane = t & 31;
    // shared-window address of plane PA / distance to PB, pinned in registers (left to itself the compiler re-derives the
    // window base from %cgaid at every use)
    uint32_t pa_s = smem_u32(PA), pb_off = (uint32_t)((const char*)PB - (const char*)PA);
    asm volatile("" : "+r"(pa_s), "+r"(pb_off));
    VAR_GROUP_LOOP(grp, B, G, t) {
        const VarGroup V = var_group(g, B, grp);
        const uint32_t* __restrict__ fw = reinterpret_cast<const uint32_t*>(g.vfwd + B.t0 + V.base) + lane;   // row pair k: fw[32 k]
        int b = B.b0;
        bool runs = V.have;
        uint32_t stk = stk_blk;
        if (MULTI) {
            if (V.have) {
                b = g.bvm[V.i]; runs = blk_problem_runs(s, b); stk = (runs && s.nanflag[b]) ? 0x80000000u : 0u;
                if (!runs) for (int j = 0; j < V.deg; ++j) PA[(fw[32 * (j >> 1)] >> (16 * (j & 1))) & 0x7fffu] = __uint_as_float(PDP_SLOT_SKIP);
            }
        }
        if (!runs) continue;
        const uint32_t act = (uint32_t)s.av[V.i];
        float P = 0.f, N = 0.f, n0 = 0.f, d0 = 0.f, n1 = 0.f, d1 = 0.f;
        // Rows go two at a time: both rows' shared-memory reads, then their arithmetic (two independent chains), then their
        // writes.  (Row by row the compiler cannot move the reads of one row above the write of the row before -- the planes
        // are indexed through the table -- and the logarithm chains of a warp run back to back.)  The table entries are
        // fetched four rows ahead: global memory, the CTAs leave no L1 to speak of.
        // table entries: one 32-bit word per row pair, fetched two pairs (four rows) ahead
        const int npair = (V.deg + 1) >> 1;
        uint32_t eq[2];
#pragma unroll
        for (int k = 0; k < 2; ++k) eq[k] = (k < npair) ? fw[32 * k] : 0u;
        auto stat_row = [&](uint32_t en, uint32_t nb, float xo, float y) {
            const float xn = __uint_as_float(nb & 0x7fffffffu);
            if (en >> 15) N += y; else P += y;          // (the reference adds 0 * y to the other sum: x + 0 = x, see above for NaN)
            const float c = X30S(xn);
            n0 += xn * c; d0 += c;
            if (PREV) {
                float d = fabsf(xo - xn);
                if (MASKED && em_set && (int32_t)nb < 0) d = d * 0.f;
                const float cd = X30S(d);
                n1 += d * cd; d1 += cd;
            }
        };
        for (int k0 = 0; k0 < npair; k0 += 2) {
#pragma unroll
            for (int h = 0; h < 2; ++h) {
                const int k = k0 + h;
                if (k >= npair) break;
                const bool vb = 2 * k + 1 < V.deg;
                const uint32_t ew = eq[h];
                if (k + 2 < npair) eq[h] = fw[32 * (k + 2)];
                const uint32_t ea = ew & 0xffffu, eb = vb ? (ew >> 16) : ea;
                const uint32_t aa = pa_s + ((ea & 0x7fffu) << 2), ab = pa_s + ((eb & 0x7fffu) << 2);
                const uint32_t nba = lds_u32(aa); const float xoa = lds_f32(aa + pb_off);
                const uint32_t nbb = lds_u32(ab); const float xob = lds_f32(ab + pb_off);
                float ya = L40_1m(xoa), yb = L40_1m(xob);
                if (MASKED && use_mask && (int32_t)nba < 0) ya = ya * 0.f;      // edge masked
                if (MASKED && use_mask && (int32_t)nbb < 0) yb = yb * 0.f;
                sts_f32(aa + pb_off, ya);
                if (vb) sts_f32(ab + pb_off, yb);
                stat_row(ea, nba, xoa, ya);
                if (vb) stat_row(eb, nbb, xob, yb);
            }
        }
        {
            const float sm0 = pdp_divs(n0, tmaxf(d0, 1.0f)) * (float)act;
            const float sm1 = pdp_divs(n1, tmaxf(d1, 1.0f)) * (float)act;
            if (!MULTI) {
                red.touch(s, b);
                red.acc.add(sm0, sm1, PREV, act);
            } else {
                StatAcc one;
                one.reset();
                one.add(sm0, sm1, PREV, act);
                if (local_stats) {
                    const int lb = b - B.b0;
                    atomicMax(&sm_st.mx0[lb], one.mx0); atomicMin(&sm_st.mn0[lb], one.mn0);
                    if (PREV) { atomicMax(&sm_st.mx1[lb], one.mx1); atomicMin(&sm_st.mn1[lb], one.mn1); }
                    if (one.nan) atomicOr(&sm_st.nan[lb], one.nan);
                    if (act) atomicAdd(&sm_st.nav[lb], act);
                } else {
                    one.commit(s, b);
                }
            }
        }
        float sb_pos, opp_pos, O_pos, sb_neg, opp_neg, O_neg, l_pos = 0.f, l_neg = 0.f;
        if (REINF) {
            const float e = s.ext[g.var_ptr[V.i]];
            l_pos = L40(1.0f - pi * ((e == 1.f) ? 1.f : 0.f));    // same of s = +1, opp of s = -1
            l_neg = L40(1.0f - pi * ((e == -1.f) ? 1.f : 0.f));   // same of s = -1, opp of s = +1
            sp_var_prepare_pi(P, N, 1.f, l_neg, sb_pos, opp_pos, O_pos);
            sp_var_prepare_pi(P, N, -1.f, l_pos, sb_neg, opp_neg, O_neg);
        } else {
            sp_var_prepare(P, N, 1.f, sb_pos, opp_pos, O_pos);
            sp_var_prepare(P, N, -1.f, sb_neg, opp_neg, O_neg);
        }
        bool made_nan = false;
#pragma unroll
        for (int k = 0; k < 2; ++k) eq[k] = (k < npair) ? fw[32 * k] : 0u;
        // q <= 1 (total >= u) or NaN: bit 30 of the results' OR tells whether a NaN was produced.  (A q >= 2 out of surveys
        // that are no probabilities sets it as well: the problem then takes the sticky path for nothing, same results.)
        uint32_t nan_or = 0u;
        auto fin_row = [&](uint32_t en, float y) {
            const bool neg = (en >> 15) != 0u;
            if (REINF) return sp_var_finish_pi(neg ? sb_neg : sb_pos, neg ? l_neg : l_pos, neg ? opp_neg : opp_pos, neg ? O_neg : O_pos, y);
            return sp_var_finish(neg ? sb_neg : sb_pos, neg ? opp_neg : opp_pos, neg ? O_neg : O_pos, y);
        };
        for (int k0 = 0; k0 < npair; k0 += 2) {
#pragma unroll
            for (int h = 0; h < 2; ++h) {
                const int k = k0 + h;
                if (k >= npair) break;
                const bool vb = 2 * k + 1 < V.deg;
                const uint32_t ew = eq[h];
                if (k + 2 < npair) eq[h] = fw[32 * (k + 2)];
                const uint32_t ea = ew & 0xffffu, eb = vb ? (ew >> 16) : ea;
                const uint32_t aa = pa_s + ((ea & 0x7fffu) << 2), ab = pa_s + ((eb & 0x7fffu) << 2);
                const float ya = lds_f32(aa + pb_off), yb = lds_f32(ab + pb_off);
                const uint32_t ua = __float_as_uint(fin_row(ea, ya)), ub = __float_as_uint(fin_row(eb, yb));
                nan_or |= ua | ub;     // (row b of an odd tail repeats row a)
                sts_u32(aa, ua | stk);
                if (vb) sts_u32(ab, ub | stk);
            }
        }
        made_nan = (nan_or & 0x40000000u) != 0u;
        if (made_nan) s.nanpend[b] = 1;
    }
}

__device__ __forceinline__ void stats_slots_reset(BlkStats& sm_st, int t, int nprob) {
    if (t < nprob) {
        sm_st.mx0[t] = 0u; sm_st.mn0[t] = 0x7f800000u; sm_st.mx1[t] = 0u; sm_st.mn1[t] = 0x7f800000u;
        sm_st.nan[t] = 0u; sm_st.nav[t] = 0u;
    }
}
__device__ __forceinline__ void stats_slots_commit(const pdp_state& s, BlkStats& sm_st, int t, int nprob, int b0) {
    if (t < nprob) {
        StatAcc a;
        a.mx0 = sm_st.mx0[t]; a.mn0 = sm_st.mn0[t]; a.mx1 = sm_st.mx1[t]; a.mn1 = sm_st.mn1[t];
        a.nan = sm_st.nan[t]; a.nav = sm_st.nav[t];
        if (a.mn0 != 0x7f800000u || a.mx0 != 0u || a.nan || a.nav || a.mn1 != 0x7f800000u) a.commit(s, b0 + t);
    }
}

// PDP_PHASE_TIMING (profiling builds only): thread 0 of every CTA adds the clock cycles (>> 10) it spent in each
// phase of the blocked passes to the trace buffer: [0..2] clause load / node / write-out, [3..5] variable
#ifdef PDP_PHASE_TIMING
#define PHASE_T0() long long _pt = clock64()
#define PHASE_ADD(slot_) do { if (threadIdx.x == 0 && A.trace) { const long long _n = clock64(); atomicAdd(&A.trace[slot_], (int)((_n - _pt) >> 10)); _pt = _n; } } while (0)
#else
#define PHASE_T0() do {} while (0)
#define PHASE_ADD(slot_) do {} while (0)
#endif

// Block hand-out of one pass.  Static (block b to CTA b mod grid) when one CTA owns the SM: the CTAs then finish within
// 1-2 % of each other.  With two CTAs per SM the pair drifts apart, the early one waits at the grid barrier and its
// partner finishes alone at half the SM's warps (10 % of the iteration, measured), so the blocks after a CTA's first one
// come from a counter.  Nothing on the way to a block's bulk copies may wait for global memory: the counter is read TWO
// blocks ahead (thread 0 picks up, at the top of a block, the ticket it drew at the top of the block before and draws the
// next one), and the descriptor of the next block is fetched during the current block's write-out and handed over in
// shared memory (NextBlk).
struct Feeder {
    int pending;    // (thread 0) ticket drawn at the top of the previous block: index of the block after the next one
};
template <bool DYN>
__device__ __forceinline__ int feed_draw(int* ctr, int blk_static) {
    return DYN ? (int)gridDim.x + atomicAdd(ctr, 1) : blk_static;
}
// all threads, after the block's last use of shared memory
__device__ __forceinline__ int feed_advance(const int* slot, int& par) {
    __syncthreads();
    const int nx = slot[par];
    par ^= 1;
    return nx;
}

// Two CTAs share an SM so that one's memory phases (load, write-out: DRAM latency, idle issue slots) overlap the other's
// node phase (issue bound, no DRAM traffic).  Both leave a grid barrier at the same time, and with equal blocks they
// would then run the same phase at the same time for the whole pass: the second CTA of an SM starts a pass about half a
// block period late.
__device__ __forceinline__ void blk_stagger(int sm_rank, int cycles) {
    if (sm_rank == 0 || cycles <= 0) return;
    const long long t0 = clock64();
    while (clock64() - t0 < cycles) __nanosleep(256);
}

// thread 0: will the blocked pass process block N?  1 yes, 2 no, 0 not looked at (a block of very many problems)
__device__ __forceinline__ int blk_will_run(const pdp_state& s, const BlkGeo& N) {
    if (N.n1 <= N.n0 || N.ne <= 0) return 2;
    if (N.b1 - N.b0 >= 128) return 0;
    for (int b = N.b0; b <= N.b1; ++b) if (blk_problem_runs(s, b)) return 1;
    return 2;
}
// The descriptor of the block a CTA takes next is fetched (by thread 0, while the CTA waits for the current block's copies)
// and handed over in shared memory: at the top of the next block nothing stands between the barrier and the bulk copies.
struct NextBlk {
    BlkGeo B;
    int blk;        // the block B describes (-1: nothing)
    int state;      // blk_will_run
};

// state of the CTA's bulk-copy barrier: one mbarrier for the kernel's lifetime, its phase parity carried in a register
struct BulkBar {
    uint64_t* bar;
    uint32_t parity;
};

// clause pass of iteration t: eta(t) [buffer r^1, V-layout] from q(t-1) [C-layout]
template <int CTAS>
__device__ __forceinline__ void blk_clause_pass(const KArgs& A, int r, bool use_mask, unsigned char* smem, int sm_rank, BulkBar& bb) {
    using Cfg = SweepCfg<CTAS>;
    constexpr int NT = Cfg::kThreads, CAP = Cfg::kAdjCap;
    const pdp_graph& g = A.g; const pdp_state& s = A.s;
    float* X0 = reinterpret_cast<float*>(smem);
    uint2* wrun_s = reinterpret_cast<uint2*>(smem + Cfg::kPlaneBytes);
    int32_t* adj_s = reinterpret_cast<int32_t*>(smem + Cfg::kPlaneBytes + 8 * Cfg::kRunWords);
    const float* __restrict__ qin = s.qu;
    float* __restrict__ eout = s.eta[r ^ 1];
    const int tid = threadIdx.x;
    __shared__ int sm_feed[2];
    __shared__ NextBlk sm_next[2];
    constexpr bool DYN = CTAS == 2;
    int par = 0;
    Feeder fd;
    fd.pending = (tid == 0) ? feed_draw<DYN>(&s.ctrl[CTRL_NEXT_CBLK], (int)blockIdx.x + (int)gridDim.x) : 0;
    if (tid < 2) sm_next[tid].blk = -1;
    __syncthreads();
    if (CTAS == 2) blk_stagger(sm_rank, A.stagger_c);
    for (int blk = blockIdx.x; blk < g.ncb; blk = feed_advance(sm_feed, par)) {
        int nx = 0;      // (thread 0) the block after this one
        if (tid == 0) {
            nx = fd.pending;
            fd.pending = feed_draw<DYN>(&s.ctrl[CTRL_NEXT_CBLK], nx + (int)gridDim.x);
            sm_feed[par] = nx;
        }
        BlkGeo B;
        int known = 0;
        if (sm_next[par ^ 1].blk == blk) { B = sm_next[par ^ 1].B; known = sm_next[par ^ 1].state; }
        else B = clause_block(g, blk);
        if (known == 2) continue;
        if (known == 0) {
            if (B.n1 <= B.n0 || B.ne <= 0) continue;
            if (blk_idle(s, B.b0, B.b1)) continue;
        }
        PHASE_T0();
        const BlkStage S = blk_stage<CAP>(B);
        if (tid == 0) {
            fence_proxy_async_smem();      // the previous block's generic-proxy accesses of the planes precede these copies
            mbar_expect_tx(bb.bar, (uint32_t)(S.nbytes + S.wbytes + S.rbytes));
            bulk_g2s(X0, qin + S.a0, S.nbytes, bb.bar);
            bulk_g2s(wrun_s, g.c_wrun + S.w0, S.wbytes, bb.bar);
            if (S.rbytes) bulk_g2s(adj_s, g.c_wadj + S.r0, S.rbytes, bb.bar);
        }
        float* X = X0 + S.shift;
        const bool masked = use_mask && (B.multi() || s.masked[B.b0]);
        const uint32_t stk_blk = (!B.multi() && s.nanflag[B.b0]) ? 0x80000000u : 0u;
        const int ku = g.cb_k[blk];
        MaskWords MW; MW.m0 = 0u; MW.m1 = 0u;
        if (masked) MW = ph_mask_fetch<NT>(tid, g.qmask, B);
        mbar_wait_cta(bb.bar, bb.parity);
        bb.parity ^= 1u;
        if (masked) { ph_apply_mask<NT>(tid, g.qmask, B, X, MW); __syncthreads(); }
        PHASE_ADD(0);
        if (masked) ph_clause_node<NT, true>(tid, g, s, B, ku, X, stk_blk);
        else ph_clause_node<NT, false>(tid, g, s, B, ku, X, stk_blk);
        __syncthreads();
        PHASE_ADD(1);
        ph_write_out<NT>(tid, B, B.e0, B.e0 + B.ne, X, wrun_s, S.w0, S.rbytes ? adj_s : nullptr, S.r0, g.c_wadj, s.eta[r], eout, B.multi() || stk_blk != 0u);
        // meanwhile thread 0 looks at the next block: its descriptor for the hand-over, its tables -> L2 (the tables only:
        // pulling the messages in as well loses 3 % on 8 x n = 1M -- the regions of 296 CTAs crowd each other out of L2)
        if (tid == 0 && nx < g.ncb) {
            const BlkGeo N = clause_block(g, nx);
            sm_next[par].B = N; sm_next[par].blk = nx; sm_next[par].state = blk_will_run(s, N);
            if (N.ne > 0) {
                bulk_prefetch_l2(g.cfwd + N.t0, 2 * N.tn);
                bulk_prefetch_l2(g.c_wrun + (N.e0 >> 5), 8 * (N.ne / 32 + 2));
                bulk_prefetch_l2(g.c_wadj + N.run0, 4 * N.nruns);
            }
        }
        PHASE_ADD(2);
    }
    fence_proxy_async();   // this pass's stores precede the bulk copies of the next pass (other CTAs, after the grid barrier)
}

// variable pass of iteration t: the decimator statistics of eta(t) [buffer r^1] against eta(t-1)
// [buffer r], and q(t) [C-layout, in place] from eta(t-1)
template <int CTAS, bool REINF>
__device__ __forceinline__ void blk_var_pass(const KArgs& A, int r, bool use_mask, bool has_prev, bool em_set, unsigned char* smem, int sm_rank, BulkBar& bb) {
    using Cfg = SweepCfg<CTAS>;
    constexpr int NT = Cfg::kThreads, CAP = Cfg::kAdjCap;
    const pdp_graph& g = A.g; const pdp_state& s = A.s;
    float* PA0 = reinterpret_cast<float*>(smem);   // eta(t), then q(t)
    float* PB0 = PA0 + Cfg::kPlaneV;               // eta(t-1), then y
    uint2* wrun_s = reinterpret_cast<uint2*>(smem + Cfg::kPlaneBytes);
    int32_t* adj_s = reinterpret_cast<int32_t*>(smem + Cfg::kPlaneBytes + 8 * Cfg::kRunWords);
    __shared__ BlkStats sm_st;
    const float* __restrict__ en = s.eta[r ^ 1];
    const float* __restrict__ eo = s.eta[r];
    const int tid = threadIdx.x;
    KeyedReducer<StatAcc> red;
    int acc_key = -1;
    __shared__ int sm_feed[2];
    __shared__ NextBlk sm_next[2];
    constexpr bool DYN = CTAS == 2;
    int par = 0;
    Feeder fd;
    fd.pending = (tid == 0) ? feed_draw<DYN>(&s.ctrl[CTRL_NEXT_VBLK], (int)blockIdx.x + (int)gridDim.x) : 0;
    if (tid < 2) sm_next[tid].blk = -1;
    __syncthreads();
    if (CTAS == 2) blk_stagger(sm_rank, A.stagger_v);
    for (int blk = blockIdx.x; blk < g.nvb; blk = feed_advance(sm_feed, par)) {
        int nx = 0;
        if (tid == 0) {
            nx = fd.pending;
            fd.pending = feed_draw<DYN>(&s.ctrl[CTRL_NEXT_VBLK], nx + (int)gridDim.x);
            sm_feed[par] = nx;
        }
        BlkGeo B;
        int known = 0;
        if (sm_next[par ^ 1].blk == blk) { B = sm_next[par ^ 1].B; known = sm_next[par ^ 1].state; }
        else B = var_block(g, blk);
        if (known == 2) continue;
        if (known == 0) {
            if (B.n1 <= B.n0 || B.ne <= 0) continue;
            if (blk_idle(s, B.b0, B.b1)) continue;
        }
        PHASE_T0();
        const BlkStage S = blk_stage<CAP>(B);
        if (tid == 0) {
            fence_proxy_async_smem();
            mbar_expect_tx(bb.bar, (uint32_t)(2 * S.nbytes + S.wbytes + S.rbytes));
            bulk_g2s(PB0, eo + S.a0, S.nbytes, bb.bar);
            bulk_g2s(PA0, en + S.a0, S.nbytes, bb.bar);
            bulk_g2s(wrun_s, g.v_wrun + S.w0, S.wbytes, bb.bar);
            if (S.rbytes) bulk_g2s(adj_s, g.v_wadj + S.r0, S.rbytes, bb.bar);
        }
        float* PA = PA0 + S.shift;
        float* PB = PB0 + S.shift;
        const bool local_stats = B.multi() && (B.b1 - B.b0 < PDP_STAT_SLOTS);   // else: registers (one problem) or global atomics
        // statistics of single-problem blocks: the per-thread accumulators run across the blocks of one problem and are
        // merged block-wide when the CTA moves on to another problem (and at the end of the pass)
        if (!B.multi() && acc_key != B.b0) { if (acc_key >= 0) red.finish(s); acc_key = B.b0; }
        if (local_stats) stats_slots_reset(sm_st, tid, B.b1 - B.b0 + 1);
        const bool masked = (use_mask || em_set) && (B.multi() || s.masked[B.b0]);
        const uint32_t stk_blk = (!B.multi() && s.nanflag[B.b0]) ? 0x80000000u : 0u;
        const bool scoring = !REINF && (s.want_score[B.b0] || s.want_score[B.b1]);
        MaskWords MW; MW.m0 = 0u; MW.m1 = 0u;
        if (masked) MW = ph_mask_fetch<NT>(tid, g.vmask, B);
        mbar_wait_cta(bb.bar, bb.parity);
        bb.parity ^= 1u;
        if (masked) ph_apply_mask<NT>(tid, g.vmask, B, PA, MW);
        if (masked) __syncthreads();      // (the per-problem statistics slots were reset before the wait's barrier)
        PHASE_ADD(3);
        // SurveyScorer of problems about to converge, while the new surveys are still in the plane (the node phase
        // overwrites them); its own loop, so that the node phase's code is the same with and without it
        if (scoring) { ph_var_score<NT>(tid, g, s, B, PA); __syncthreads(); }
        {
#define VN_CALL(MU, MA, PR) ph_var_node<NT, MU, MA, PR, REINF>(tid, g, s, B, use_mask, em_set, PA, PB, stk_blk, red, sm_st, local_stats, A.rf.pi)
            if (B.multi()) { if (has_prev) VN_CALL(true, true, true); else VN_CALL(true, true, false); }
            else if (masked) { if (has_prev) VN_CALL(false, true, true); else VN_CALL(false, true, false); }
            else { if (has_prev) VN_CALL(false, false, true); else VN_CALL(false, false, false); }
#undef VN_CALL
        }
        __syncthreads();
        PHASE_ADD(4);
        if (local_stats) stats_slots_commit(s, sm_st, tid, B.b1 - B.b0 + 1, B.b0);
        ph_write_out<NT>(tid, B, B.e0, B.e0 + B.ne, PA, wrun_s, S.w0, S.rbytes ? adj_s : nullptr, S.r0, g.v_wadj, s.qu, s.qu, B.multi() || stk_blk != 0u);
        if (tid == 0 && nx < g.nvb) {      // the next block's descriptor and tables (see the clause pass)
            const BlkGeo N = var_block(g, nx);
            sm_next[par].B = N; sm_next[par].blk = nx; sm_next[par].state = blk_will_run(s, N);
            if (N.ne > 0) {
                bulk_prefetch_l2(g.vfwd + N.t0, 2 * N.tn);
                bulk_prefetch_l2(g.vsort + N.n0, 8 * (N.n1 - N.n0));
                bulk_prefetch_l2(g.v_wrun + (N.e0 >> 5), 8 * (N.ne / 32 + 2));
                bulk_prefetch_l2(g.v_wadj + N.run0, 4 * N.nruns);
            }
        }
        PHASE_ADD(5);
    }
    red.finish(s);
    fence_proxy_async();
}
