// pdp_graph.cu -- graph ingest: the reference's batch tensors -> CSR (by clause) + CSC (by variable).
// Replaces SATProblem.setup_problem and the 14 sparse COO incidence matrices it builds
// (reference pdp/nn/solver.py:28-54,101-178).  Adjacency lists are STABLE (ascending original edge
// index inside every node) because that is the fp32 accumulation order of torch.mm(sparse, dense).
#include <cub/cub.cuh>
#include <stdarg.h>

#include "pdp_common.cuh"

int pdp_build_layout(pdp_ctx* c, cudaStream_t stream, bool monotone_maps);   // pdp_layout.cu

static thread_local char g_err[512] = "";

void pdp_set_error(const char* fmt, ...) {
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(g_err, sizeof(g_err), fmt, ap);
    va_end(ap);
}

extern "C" const char* pdp_last_error(void) { return g_err; }
#ifdef PDP_STRICT_MATH
extern "C" const char* pdp_version(void) { return "pdp_b200 0.1 (sm_100a, strict-math test build)"; }
#else
extern "C" const char* pdp_version(void) { return "pdp_b200 0.1 (sm_100a)"; }
#endif

// ------------------------------------------------------------------------------------------------
// workspace carving
// ------------------------------------------------------------------------------------------------
namespace {

struct Carver {
    uint8_t* base;
    size_t off;
    bool dry;
    template <typename T>
    T* take(int64_t n) {
        size_t bytes = (size_t)(n > 0 ? n : 1) * sizeof(T);
        off = (off + 255) & ~(size_t)255;
        T* p = dry ? nullptr : reinterpret_cast<T*>(base + off);
        off += bytes;
        return p;
    }
};

size_t cub_reserve(int64_t E, int64_t V, int64_t F) {
    size_t n = (size_t)(E > V ? E : V);
    if ((size_t)F > n) n = (size_t)F;
    return (size_t)(1 << 20) + n / 2;
}

void carve(pdp_ctx* c, Carver& k, int64_t E, int64_t V, int64_t F, int64_t B) {
    pdp_graph& g = c->g;
    pdp_state& s = c->s;
    g.cl_ptr = k.take<int32_t>(F + 1);
    g.var_ptr = k.take<int32_t>(V + 1);
    g.c_orig = k.take<int32_t>(E);
    g.c_var = k.take<uint32_t>(E);
    g.c_pos = k.take<int32_t>(E);
    g.v_cedge = k.take<uint32_t>(E);
    g.v_cls = k.take<int32_t>(E);
    g.v_orig = k.take<int32_t>(E);
    g.bvm = k.take<int32_t>(V);
    g.bfm = k.take<int32_t>(F);
    g.prob_vptr = k.take<int32_t>(B + 1);
    g.prob_fptr = k.take<int32_t>(B + 1);
    g.p_vpos = k.take<int32_t>(E);
    g.p_qpos = k.take<int32_t>(E);
    g.vmask = k.take<uint32_t>(E / 32 + 1);
    g.qmask = k.take<uint32_t>(E / 32 + 1);
    // block count <= rounds * SMs + 1 with rounds * SMs <= E / (half a block) + SMs (pdp_layout.cu pick_stride;
    // nodes of degree above half a block disable the blocked path)
    const int64_t max_vb = E / (PDP_BLK_V / 4) + 2 * PDP_MAX_SMS + 2, max_cb = E / (PDP_BLK_C / 4) + 2 * PDP_MAX_SMS + 2;
    g.vb_desc = k.take<pdp_blk>(max_vb + 1);
    g.cb_desc = k.take<pdp_blk>(max_cb + 1);
    g.vb_ptr = k.take<int32_t>(max_vb + 1);
    g.cb_ptr = k.take<int32_t>(max_cb + 1);
    g.vfwd_cap = 2 * E + 64 * (max_vb + 1);   // (a block's last, partial group pads up to 31 lanes)
    g.vfwd = k.take<uint16_t>(g.vfwd_cap + 8);
    g.cfwd = k.take<uint16_t>(E + 8);
    g.vb_t0 = k.take<int32_t>(max_vb + 2);
    g.v_wrun = k.take<uint2>(E / 32 + 2);
    g.c_wrun = k.take<uint2>(E / 32 + 2);
    g.v_wadj = k.take<int32_t>(E);
    g.c_wadj = k.take<int32_t>(E);
    g.wo_tmp = k.take<int32_t>(3 * (E / 32 + 2));
    g.vsort = k.take<int2>(V);
    g.cb_k = k.take<int32_t>(max_cb + 1);
    s.eta[0] = k.take<float>(E);
    s.eta[1] = k.take<float>(E);
    s.qu = k.take<float>(E);
    s.qs = k.take<float>(E);
    s.qd = k.take<float>(E);
    s.ext = k.take<float>(E);
    s.av = k.take<uint8_t>(V);
    s.af = k.take<uint8_t>(F);
    s.sol = k.take<float>(V);
    s.is_sat = k.take<float>(B);
    s.active = k.take<uint8_t>(B);
    s.counters = k.take<int32_t>(B);
    s.freeze_iter = k.take<int32_t>(B);
    s.flags = k.take<uint32_t>(B);
    s.masked = k.take<uint8_t>(B);
    s.dirty = k.take<uint8_t>(B);
    s.conv = k.take<uint8_t>(B);
    s.nanflag = k.take<uint8_t>(B);
    s.nanpend = k.take<uint8_t>(B);
    s.st_max = k.take<uint32_t>(2 * B);
    s.st_min = k.take<uint32_t>(2 * B);
    s.st_nan = k.take<uint32_t>(B);
    s.nav = k.take<int32_t>(B);
    s.c_max = k.take<uint32_t>(B);
    s.c_min = k.take<uint32_t>(B);
    s.c_nan = k.take<uint32_t>(B);
    s.arg_idx = k.take<int32_t>(B);
    s.loc_list = k.take<int32_t>(B);
    s.n_unsat = k.take<int32_t>(B);
    s.conflicts = k.take<int32_t>(B);
    s.score = k.take<float>(V);
    s.up_cnt = k.take<int32_t>(V);
    s.up_ev = k.take<int32_t>(V);
    s.pure = k.take<uint8_t>(V);
    s.single = k.take<uint8_t>(F);
    for (int i = 0; i < 4; ++i) s.fr_list[i] = k.take<int32_t>(PDP_FR_CAP);
    for (int i = 0; i < 2; ++i) s.fr_unit[i] = k.take<int32_t>(PDP_FR_CAP);
    s.fr_cap = PDP_FR_CAP;
    if (const char* cap = getenv("PDP_B200_FR_CAP")) { const int v = atoi(cap); if (v >= 1 && v < PDP_FR_CAP) s.fr_cap = v; }
    s.want_score = k.take<uint8_t>(B);
    s.have_score = k.take<uint8_t>(B);
    s.last_d = k.take<float>(B);
    s.stamp_c = k.take<int32_t>(F);
    s.stamp_v = k.take<int32_t>(V);
    s.sel_hist = k.take<uint32_t>(B * PDP_SEL_BINS);
    s.sel_pref = k.take<unsigned long long>(B);
    s.sel_need = k.take<int32_t>(B);
    s.sel_sh = k.take<int32_t>(B);
    s.rb_h = k.take<int32_t>(B);
    s.rb_count = k.take<int32_t>(B);
    s.rb_last = k.take<int32_t>(B);
    s.rb_snap = k.take<uint8_t>(B);
    s.ctrl = k.take<int32_t>(CTRL_SIZE);
    s.sm_ctr = k.take<int32_t>(PDP_MAX_SMS);
    s.asg = k.take<int8_t>(V);
    s.ws_true = k.take<int32_t>(F);
    s.ws_deg = k.take<int32_t>(F);
    s.ws_best = k.take<uint32_t>(2 * B);
    s.ws_key = k.take<unsigned long long>(2 * B);
    s.energy = k.take<int32_t>(B);
    s.scan_tmp = k.take<int32_t>(V + 1);
    c->cub_tmp_bytes = cub_reserve(E, V, F);
    c->cub_tmp = k.take<uint8_t>((int64_t)c->cub_tmp_bytes);
}

// ------------------------------------------------------------------------------------------------
// kernels
// ------------------------------------------------------------------------------------------------
__global__ void k_check_and_count(const int32_t* __restrict__ evar, const int32_t* __restrict__ ecls, int64_t E,
                                  int64_t V, int64_t F, int32_t* cl_cnt, int32_t* var_cnt, int32_t* flags) {
    for (int64_t e = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; e < E; e += (int64_t)gridDim.x * blockDim.x) {
        int32_t v = evar[e], a = ecls[e];
        if (v < 0 || v >= V || a < 0 || a >= F) { atomicOr(&flags[1], 1); continue; }
        if (e > 0 && ecls[e - 1] > a) atomicOr(&flags[0], 1);   // not clause-major
        atomicAdd(&cl_cnt[a + 1], 1);
        atomicAdd(&var_cnt[v + 1], 1);
    }
}

__global__ void k_check_maps(const int32_t* __restrict__ bvm, const int32_t* __restrict__ bfm, int64_t V, int64_t F,
                             int64_t B, int32_t* flags) {
    int64_t n = V > F ? V : F;
    for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) {
        if (i < V && (bvm[i] < 0 || bvm[i] >= B)) atomicOr(&flags[1], 2);
        if (i < F && (bfm[i] < 0 || bfm[i] >= B)) atomicOr(&flags[1], 2);
        // the blocked sweep skips whole blocks by the problem range of their first and last node
        if (i > 0 && i < V && bvm[i - 1] > bvm[i]) atomicOr(&flags[4], 1);
        if (i > 0 && i < F && bfm[i - 1] > bfm[i]) atomicOr(&flags[4], 1);
    }
}

__global__ void k_iota(int32_t* out, int64_t n) {
    for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x)
        out[i] = (int32_t)i;
}

// inv[c_orig[c]] = c
__global__ void k_invert(const int32_t* __restrict__ perm, int32_t* inv, int64_t n) {
    for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x)
        inv[perm[i]] = (int32_t)i;
}

__global__ void k_fill_clause_major(const int32_t* __restrict__ evar, const float* __restrict__ sign,
                                    const int32_t* __restrict__ c_orig, uint32_t* c_var, int64_t E) {
    for (int64_t c = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; c < E; c += (int64_t)gridDim.x * blockDim.x) {
        int32_t e = c_orig[c];
        c_var[c] = (uint32_t)evar[e] | ((sign[e] < 0.f) ? PDP_SIGN_BIT : 0u);
    }
}

// sort payload of the variable-major order: the original edge index with the literal's sign in bit 31, so that the fill
// below does not have to gather the sign again (one random 4-byte gather per edge less)
__global__ void k_iota_signed(const float* __restrict__ sign, uint32_t* out, int64_t E) {
    for (int64_t e = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; e < E; e += (int64_t)gridDim.x * blockDim.x)
        out[e] = (uint32_t)e | ((sign[e] < 0.f) ? PDP_SIGN_BIT : 0u);
}

// packed[p] = original edge index | sign of slot p (stable sort by variable); v_orig[p] is written here
__global__ void k_fill_var_major(const int32_t* __restrict__ ecls, const uint32_t* __restrict__ packed,
                                 const int32_t* __restrict__ inv, int32_t* v_orig,
                                 uint32_t* v_cedge, int32_t* v_cls, int32_t* c_pos, int64_t E) {
    for (int64_t p = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; p < E; p += (int64_t)gridDim.x * blockDim.x) {
        const uint32_t w = packed[p];
        const int32_t e = (int32_t)(w & PDP_IDX_MASK);
        const int32_t c = inv ? inv[e] : e;
        v_orig[p] = e;
        v_cedge[p] = (uint32_t)c | (w & PDP_SIGN_BIT);
        v_cls[p] = ecls[e];
        c_pos[c] = (int32_t)p;
    }
}

__global__ void k_max_degree(const int32_t* __restrict__ ptr, int64_t n, int32_t* out) {
    int32_t m = 0;
    for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) {
        int32_t d = ptr[i + 1] - ptr[i];
        m = d > m ? d : m;
    }
    for (int o = 16; o > 0; o >>= 1) { int32_t t = __shfl_xor_sync(0xffffffffu, m, o); m = t > m ? t : m; }
    if ((threadIdx.x & 31) == 0 && m > 0) atomicMax(out, m);
}

}  // namespace

// prob_vptr[b] = first variable of problem b (lower bound of b in the non-decreasing batch_variable_map)
__global__ void k_problem_ptr(const int32_t* __restrict__ bvm, int64_t V, int64_t B, int32_t* prob_vptr) {
    for (int64_t b = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; b <= B; b += (int64_t)gridDim.x * blockDim.x) {
        int64_t lo = 0, hi = V;
        while (lo < hi) {
            const int64_t mid = (lo + hi) >> 1;
            if (bvm[mid] < b) lo = mid + 1; else hi = mid;
        }
        prob_vptr[b] = (int32_t)lo;
    }
}

__global__ void k_reset_state(pdp_graph g, pdp_state s, int64_t V, int64_t F, int64_t B) {
    int64_t n = V > F ? V : F;
    if (B > n) n = B;
    if (g.E / 32 + 1 > n) n = g.E / 32 + 1;
    for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) {
        if (i < g.E / 32 + 1) { g.vmask[i] = 0u; g.qmask[i] = 0u; }
        if (i < V) { s.av[i] = 1; s.sol[i] = 0.5f; s.up_cnt[i] = 0; s.up_ev[i] = 0; s.pure[i] = 0; s.score[i] = 0.f; s.asg[i] = 0; s.stamp_v[i] = 0; }
        if (i < F) { s.af[i] = 1; s.single[i] = 0; s.stamp_c[i] = 0; }
        if (i < B) {
            s.is_sat[i] = 0.5f; s.active[i] = 1; s.counters[i] = 0; s.freeze_iter[i] = -1; s.flags[i] = 0;
            s.masked[i] = 0; s.dirty[i] = 1; s.conv[i] = 0; s.nanflag[i] = 0; s.nanpend[i] = 0; s.n_unsat[i] = 0; s.conflicts[i] = 0;
            s.nav[i] = 0; s.arg_idx[i] = 0x7fffffff; s.energy[i] = 0; s.want_score[i] = 0; s.have_score[i] = 0; s.last_d[i] = 0.f;
            s.st_max[2 * i] = 0u; s.st_max[2 * i + 1] = 0u; s.st_min[2 * i] = 0x7f800000u; s.st_min[2 * i + 1] = 0x7f800000u;
            s.st_nan[i] = 0u; s.c_max[i] = 0u; s.c_min[i] = 0x7f800000u; s.c_nan[i] = 0u;
            s.sel_need[i] = -1; s.sel_sh[i] = 0; s.sel_pref[i] = 0ull;
            s.rb_h[i] = 0; s.rb_count[i] = 0; s.rb_last[i] = 0; s.rb_snap[i] = 0;
            for (int j = 0; j < PDP_SEL_BINS; ++j) s.sel_hist[i * PDP_SEL_BINS + j] = 0u;
        }
        if (i < CTRL_SIZE) s.ctrl[i] = (i == CTRL_NUM_ACTIVE) ? (int32_t)B
                                       : ((i == CTRL_ANY_DIRTY || i == CTRL_FR_EPC || i == CTRL_FR_EPV || i == CTRL_NATIVE) ? 1 : 0);
    }
}

extern "C" size_t pdp_workspace_bytes(int64_t E, int64_t V, int64_t F, int64_t B) {
    if (E < 0 || V < 0 || F < 0 || B < 0) return 0;
    pdp_ctx tmp;
    memset(&tmp, 0, sizeof(tmp));
    Carver k{nullptr, 0, true};
    carve(&tmp, k, E, V, F, B);
    return k.off + 256;
}

extern "C" int pdp_reset(pdp_ctx* ctx, void* stream_) {
    if (!ctx) { pdp_set_error("pdp_reset: null context"); return PDP_ERR_ARG; }
    cudaStream_t stream = (cudaStream_t)stream_;
    int64_t n = ctx->g.V > ctx->g.F ? ctx->g.V : ctx->g.F;
    if (ctx->g.B > n) n = ctx->g.B;
    if (ctx->g.E / 32 + 1 > n) n = ctx->g.E / 32 + 1;
    if (n < CTRL_SIZE) n = CTRL_SIZE;
    k_reset_state<<<pdp_grid(n, 256, ctx->num_sms), 256, 0, stream>>>(ctx->g, ctx->s, ctx->g.V, ctx->g.F, ctx->g.B);
    PDP_LAUNCH_CHECK(ctx);
    return PDP_OK;
}

extern "C" int pdp_create(pdp_ctx** out, const int32_t* d_graph_map, const float* d_edge_feature,
                          const int32_t* d_bvm, const int32_t* d_bfm, int64_t E, int64_t V, int64_t F, int64_t B,
                          void* d_workspace, size_t workspace_bytes, void* stream_) {
    if (!out) { pdp_set_error("pdp_create: out is null"); return PDP_ERR_ARG; }
    *out = nullptr;
    if (E < 0 || V < 0 || F < 0 || B < 0 || E >= (int64_t)0x7fffffff || V >= (int64_t)0x7fffffff || F >= (int64_t)0x7fffffff) {
        pdp_set_error("pdp_create: sizes out of range (E=%lld V=%lld F=%lld B=%lld; each must be < 2^31-1)",
                      (long long)E, (long long)V, (long long)F, (long long)B);
        return PDP_ERR_ARG;
    }
    if ((E > 0 && (!d_graph_map || !d_edge_feature)) || (V > 0 && !d_bvm) || (F > 0 && !d_bfm) || !d_workspace) {
        pdp_set_error("pdp_create: null input pointer");
        return PDP_ERR_ARG;
    }
    size_t need = pdp_workspace_bytes(E, V, F, B);
    if (workspace_bytes < need) {
        pdp_set_error("pdp_create: workspace too small (%zu < %zu bytes)", workspace_bytes, need);
        return PDP_ERR_WORKSPACE;
    }
    cudaStream_t stream = (cudaStream_t)stream_;
    pdp_ctx* c = new pdp_ctx();
    memset(c, 0, sizeof(*c));
    if (cudaGetDevice(&c->device) != cudaSuccess) { delete c; pdp_set_error("pdp_create: no CUDA device"); return PDP_ERR_CUDA; }
    // cudaGetDeviceProperties costs tens of milliseconds per call; two attributes are all that is needed
    int cc_major = 0, cc_minor = 0, sm_count = 0;
    if (cudaDeviceGetAttribute(&cc_major, cudaDevAttrComputeCapabilityMajor, c->device) != cudaSuccess ||
        cudaDeviceGetAttribute(&cc_minor, cudaDevAttrComputeCapabilityMinor, c->device) != cudaSuccess ||
        cudaDeviceGetAttribute(&sm_count, cudaDevAttrMultiProcessorCount, c->device) != cudaSuccess) {
        delete c; pdp_set_error("pdp_create: cudaDeviceGetAttribute failed"); return PDP_ERR_CUDA;
    }
    if (cc_major < 10) {
        delete c;
        pdp_set_error("pdp_create: device is sm_%d%d; this library is built for sm_100a only", cc_major, cc_minor);
        return PDP_ERR_UNSUPPORTED;
    }
    c->num_sms = sm_count;
    c->workspace = d_workspace;
    c->workspace_bytes = workspace_bytes;
    c->g.E = E; c->g.V = V; c->g.F = F; c->g.B = B;
    uintptr_t base = ((uintptr_t)d_workspace + 255) & ~(uintptr_t)255;
    Carver k{reinterpret_cast<uint8_t*>(base), 0, false};
    carve(c, k, E, V, F, B);
    pdp_graph& g = c->g;
    const int32_t* evar = d_graph_map;
    const int32_t* ecls = d_graph_map + E;
    const int nsm = c->num_sms;

#define CK(expr) do { cudaError_t _e = (expr); if (_e != cudaSuccess) { pdp_set_error("%s:%d: %s -> %s", __FILE__, __LINE__, #expr, cudaGetErrorString(_e)); delete c; return PDP_ERR_CUDA; } } while (0)
#define LK() do { c->launches++; cudaError_t _e = cudaGetLastError(); if (_e != cudaSuccess) { pdp_set_error("%s:%d: launch -> %s", __FILE__, __LINE__, cudaGetErrorString(_e)); delete c; return PDP_ERR_CUDA; } } while (0)

    if (V > 0) CK(cudaMemcpyAsync(g.bvm, d_bvm, sizeof(int32_t) * (size_t)V, cudaMemcpyDeviceToDevice, stream));
    if (F > 0) CK(cudaMemcpyAsync(g.bfm, d_bfm, sizeof(int32_t) * (size_t)F, cudaMemcpyDeviceToDevice, stream));
    CK(cudaMemsetAsync(g.cl_ptr, 0, sizeof(int32_t) * (size_t)(F + 1), stream));
    CK(cudaMemsetAsync(g.var_ptr, 0, sizeof(int32_t) * (size_t)(V + 1), stream));
    CK(cudaMemsetAsync(c->s.ctrl, 0, sizeof(int32_t) * CTRL_SIZE, stream));
    int32_t* flags = c->s.ctrl;   // [0] not clause-major, [1] index out of range, [2] max var deg, [3] max clause deg
    if (E > 0) {
        k_check_and_count<<<pdp_grid(E, 256, nsm), 256, 0, stream>>>(evar, ecls, E, V, F, g.cl_ptr, g.var_ptr, flags);
        LK();
    }
    k_check_maps<<<pdp_grid(V > F ? V : F, 256, nsm), 256, 0, stream>>>(d_bvm, d_bfm, V, F, B, flags);
    LK();
    // counts -> pointers (in-place inclusive of the leading zero = exclusive scan shifted by one)
    {
        size_t tb = c->cub_tmp_bytes;
        size_t q = 0;
        CK(cub::DeviceScan::InclusiveSum(nullptr, q, g.cl_ptr, g.cl_ptr, (int)(F + 1), stream));
        if (q > tb) { pdp_set_error("pdp_create: scan scratch %zu > reserve %zu", q, tb); delete c; return PDP_ERR_WORKSPACE; }
        CK(cub::DeviceScan::InclusiveSum(c->cub_tmp, tb, g.cl_ptr, g.cl_ptr, (int)(F + 1), stream));
        c->launches++;
        tb = c->cub_tmp_bytes;
        CK(cub::DeviceScan::InclusiveSum(c->cub_tmp, tb, g.var_ptr, g.var_ptr, (int)(V + 1), stream));
        c->launches++;
    }
    int32_t hflags[5] = {0, 0, 0, 0, 0};
    CK(cudaMemcpyAsync(hflags, flags, sizeof(hflags), cudaMemcpyDeviceToHost, stream));
    CK(cudaStreamSynchronize(stream));
    if (hflags[1]) {
        pdp_set_error("pdp_create: graph_map / batch maps hold indices outside [0,V) x [0,F) x [0,B) (code %d)", hflags[1]);
        delete c;
        return PDP_ERR_ARG;
    }
    const bool clause_major = (hflags[0] == 0);
    const bool monotone_maps = (hflags[4] == 0);

    if (E > 0) {
        // scratch aliases: message buffers are not live yet
        int32_t* kA = reinterpret_cast<int32_t*>(c->s.eta[0]);
        int32_t* kB = reinterpret_cast<int32_t*>(c->s.eta[1]);
        int32_t* vA = reinterpret_cast<int32_t*>(c->s.qu);
        int32_t* vB = reinterpret_cast<int32_t*>(c->s.qs);
        int32_t* inv = reinterpret_cast<int32_t*>(c->s.qd);
        const int32_t* sorted_vals = nullptr;   // where the last stable_sort left its payload
        // out_vals == nullptr: the payload stays in the scratch buffer (sorted_vals); signed_payload: edge index | sign bit
        auto stable_sort = [&](const int32_t* keys, int64_t nkeys, int32_t* out_vals, bool signed_payload) -> int {
            int bits = 1;
            while (((int64_t)1 << bits) < nkeys && bits < 31) ++bits;
            cudaError_t e1 = cudaMemcpyAsync(kA, keys, sizeof(int32_t) * (size_t)E, cudaMemcpyDeviceToDevice, stream);
            if (e1 != cudaSuccess) return -1;
            if (signed_payload) k_iota_signed<<<pdp_grid(E, 256, nsm), 256, 0, stream>>>(d_edge_feature, reinterpret_cast<uint32_t*>(vA), E);
            else k_iota<<<pdp_grid(E, 256, nsm), 256, 0, stream>>>(vA, E);
            c->launches++;
            cub::DoubleBuffer<int32_t> dk(kA, kB);
            cub::DoubleBuffer<int32_t> dv(vA, vB);
            size_t q = 0;
            if (cub::DeviceRadixSort::SortPairs(nullptr, q, dk, dv, (int)E, 0, bits, stream) != cudaSuccess) return -1;
            if (q > c->cub_tmp_bytes) return -2;
            size_t tb = c->cub_tmp_bytes;
            if (cub::DeviceRadixSort::SortPairs(c->cub_tmp, tb, dk, dv, (int)E, 0, bits, stream) != cudaSuccess) return -1;
            c->launches++;
            sorted_vals = dv.Current();
            if (out_vals && cudaMemcpyAsync(out_vals, dv.Current(), sizeof(int32_t) * (size_t)E, cudaMemcpyDeviceToDevice, stream) != cudaSuccess) return -1;
            return 0;
        };
        if (clause_major) {
            k_iota<<<pdp_grid(E, 256, nsm), 256, 0, stream>>>(g.c_orig, E);
            LK();
        } else {
            int r = stable_sort(ecls, F, g.c_orig, false);
            if (r != 0) { pdp_set_error("pdp_create: clause sort failed (%d)", r); delete c; return r == -2 ? PDP_ERR_WORKSPACE : PDP_ERR_CUDA; }
        }
        {
            int r = stable_sort(evar, V, nullptr, true);
            if (r != 0) { pdp_set_error("pdp_create: variable sort failed (%d)", r); delete c; return r == -2 ? PDP_ERR_WORKSPACE : PDP_ERR_CUDA; }
        }
        const uint32_t* packed = reinterpret_cast<const uint32_t*>(sorted_vals);   // vA or vB: not touched until the fill below
        if (!clause_major) {
            k_invert<<<pdp_grid(E, 256, nsm), 256, 0, stream>>>(g.c_orig, inv, E);
            LK();
        }
        k_fill_clause_major<<<pdp_grid(E, 256, nsm), 256, 0, stream>>>(evar, d_edge_feature, g.c_orig, g.c_var, E);
        LK();
        k_fill_var_major<<<pdp_grid(E, 256, nsm), 256, 0, stream>>>(ecls, packed, clause_major ? nullptr : inv, g.v_orig,
                                                                     g.v_cedge, g.v_cls, g.c_pos, E);
        LK();
        if (V > 0) { k_max_degree<<<pdp_grid(V, 256, nsm), 256, 0, stream>>>(g.var_ptr, V, flags + 2); LK(); }
        if (F > 0) { k_max_degree<<<pdp_grid(F, 256, nsm), 256, 0, stream>>>(g.cl_ptr, F, flags + 3); LK(); }
        CK(cudaMemcpyAsync(hflags, flags, sizeof(hflags), cudaMemcpyDeviceToHost, stream));
        CK(cudaStreamSynchronize(stream));
        g.max_var_degree = hflags[2];
        g.max_clause_degree = hflags[3];
    }
    g.contiguous_problems = monotone_maps ? 1 : 0;
    k_problem_ptr<<<pdp_grid(B + 1, 256, nsm), 256, 0, stream>>>(g.bvm, V, B, g.prob_vptr);
    LK();
    k_problem_ptr<<<pdp_grid(B + 1, 256, nsm), 256, 0, stream>>>(g.bfm, F, B, g.prob_fptr);
    LK();
    {
        int lrc = pdp_build_layout(c, stream, monotone_maps);
        if (lrc != PDP_OK) { delete c; return lrc; }
    }
    int rc = pdp_reset(c, stream);
    if (rc != PDP_OK) { delete c; return rc; }
#undef CK
#undef LK
    *out = c;
    return PDP_OK;
}

extern "C" int pdp_destroy(pdp_ctx* ctx) {
    delete ctx;
    return PDP_OK;
}

extern "C" int64_t pdp_launch_count(pdp_ctx* ctx) { return ctx ? ctx->launches : 0; }
