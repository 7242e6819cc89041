// pdp_edge_nn.cu -- the dense per-edge layers of the neural model types (p-nd-np, np-nd-np) on the 5th-generation tensor
// cores: tcgen05.mma (kind::tf32) issued by one thread per CTA, accumulators in tensor memory, operands in shared memory.
//
//   pdp_edge_mlp_forward   out[e, :] = act(A[e, :] W^T + b) * mask[e]          one dense layer over edge (or node) rows
//   pdp_edge_gru_forward   h'[e, :]  = GRUCell([x | feature], h)[e, :]         torch.nn.GRUCell, gates fused in the epilogue
//
// replace the nn.Linear / nn.GRUCell calls of MessageAggregator.forward (reference pdp/nn/util.py:51-77),
// NeuralDecimator.forward (pdp_decimate.py:51-87), NeuralMessagePasser.forward (pdp_propagate.py:47-95) and
// NeuralPredictor.forward (pdp_predict.py:49-91).  A row's input is the concatenation of up to three row-major sources
// (message state | edge feature | hidden state): no torch.cat copy is ever made.
//
// Precision.  The reference is fp32; one tf32 product has 11 significant bits.  Every product is therefore taken three
// times (A_hi B_hi + A_lo B_hi + A_hi B_lo with x_hi = x truncated to tf32, x_lo = x - x_hi truncated to tf32): the
// dropped terms are below 2^-21 of the product, the accumulation is fp32 in tensor memory.
//
// One CTA per SM, persistent over tiles of 128 rows.  Per tile and N-pass (<= 256 accumulator columns; the accumulator is
// double-buffered in the 512 columns of tensor memory, so the epilogue of one pass runs under the MMAs of the next), K
// goes by in chunks of 16 through a ring of shared-memory stages:
//   warps 0-7  stage the A chunk: two threads per row, each reads 8 floats of it (64-bit loads where the sources allow,
//              the next chunks' loads in flight while the current one is converted; row-strided, so they live on L1 hits --
//              a coalesced variant with eight lanes per row chunk -- 64-bit loads of four rows per warp instruction -- measured
//              20 % slower for the GRU cell and 30 % slower for the small layers), splits them, writes the hi and lo
//              operand tiles in the canonical K-major layout of the tensor core (8-row x 16-byte core matrices; 16-byte
//              column group g of a tile of R rows at g * 16 R, row r of it at + 16 r: core matrices contiguous, SBO = 128 B,
//              LBO = 16 R);
//   warp 17    one thread brings the chunk's weights with ONE bulk-asynchronous copy: the host side stores W pre-split and
//              pre-tiled, chunk after chunk, exactly as the shared-memory image (pdp_solver_b200/nn/tensor_ops.py);
//   warps 16, 18  one thread each, in turn, issues a chunk's tcgen05.mma (2 k-steps x 3 terms x N-blocks) and commits them to the stage's
//              `empty` barrier; after the pass's last chunk it commits to the accumulator buffer's barrier;
//   warps 8-15 epilogue: tcgen05.ld of the accumulator rows (thread = row, two warps per lane quadrant), bias / activation /
//              GRU gate arithmetic, 64-bit stores; then hand the accumulator buffer back.
#include <cuda_runtime.h>
#include <stdint.h>
#include <stdlib.h>

#include "pdp_common.cuh"

namespace {

constexpr int kTileM = 128;        // rows per tile = accumulator lanes
constexpr int kChunkK = 16;        // K elements per stage: one 64-byte row of the swizzled operand tiles, two MMA k-steps
                                   // (32 halves the per-chunk barrier traffic but leaves two stages: measured 20 % slower)
constexpr int kHalfK = kChunkK / 2;       // elements of a row chunk per producer thread (two threads per row)
constexpr int kThreads = 608;      // warps 0-7 A producers, 8-15 epilogue (lane quadrant = warp mod 4), 16 and 18 MMA issuers, 17 B producer
#ifndef PDP_NN_RAW_DEPTH
#define PDP_NN_RAW_DEPTH 6
#endif
constexpr int kRawDepth = PDP_NN_RAW_DEPTH;            // chunks of operand rows in flight per producer thread (cp.async ring, 8 KB each)
constexpr int kRawBytes = kRawDepth * 256 * kHalfK * 4;
constexpr int kMaxChunks = 64;                          // K <= 1024
constexpr int kMaxNTot = 320;      // accumulator columns per pass.  Two buffers in the 512 columns of tensor memory: at 0 and 256
                                   // when a pass has <= 256 columns; wider passes (the GRU cell: 4 gates x 76 units = 304) put the
                                   // second buffer at 512 - n_tot, and the columns the two share are drained first (see the epilogue)
constexpr int kMmaN = 256;         // widest tcgen05.mma: a wider pass takes two per k-step and term

enum { EPI_LINEAR = 0, EPI_GRU = 1 };
enum { ACT_NONE = 0, ACT_LOGSIGMOID = 1 };

struct EdgeNNArgs {
    const float* src[3];       // row-major sources of the A rows, concatenated along K
    int32_t ks[3];             // their column counts (0: unused)
    int32_t k_total;           // sum of ks
    int32_t k_chunks;          // ceil(k_total / 16)
    int64_t rows;              // E
    const float* w_img;        // weights, split and tiled: [pass][chunk]{hi [4][n_tot][4], lo [4][n_tot][4]}
    const float* bias;         // LINEAR: [passes * n_tot]; GRU: [passes][n_tot / 4 units][4] = r, z, i_n, h_n of every unit
    int32_t n_blk;             // (as passed: n_tot = n_blk * n_mma)
    int32_t n_mma;
    int32_t n_tot;             // accumulator columns per pass (multiple of 16, <= kMaxNTot): MMAs of kMmaN columns + the rest
    int32_t passes;
    int32_t n_out;             // LINEAR: output columns (<= passes * n_tot); GRU: hidden size H
    int32_t act;               // LINEAR
    const float* row_mask;     // [rows] or null: LINEAR multiplies the output; GRU blends mask * h' + (1 - mask) * h
    const float* h_old;        // GRU: [rows, H] (also source 0 of A)
    float* out;                // [rows, n_out]
    int32_t stages;
    int32_t out_tile;          // LINEAR: the tile's results are collected in shared memory and leave with one bulk store
};

// ---- PTX wrappers -------------------------------------------------------------------------------------------------
__device__ __forceinline__ uint32_t s_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }
__device__ __forceinline__ void mb_init(uint64_t* b, int count) { asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(s_u32(b)), "r"(count) : "memory"); }
__device__ __forceinline__ void mb_arrive(uint64_t* b) { asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(s_u32(b)) : "memory"); }
__device__ __forceinline__ void mb_expect_tx(uint64_t* b, uint32_t bytes) { asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(s_u32(b)), "r"(bytes) : "memory"); }
// SLEEP: the waiting warp backs off between polls.  The one thread that issues the MMAs shares its scheduler with four
// other warps; warps that spin on a barrier would take most of that scheduler's issue slots away from it.
template <bool SLEEP = true>
__device__ __forceinline__ void mb_wait(uint64_t* b, uint32_t parity) {
    const uint32_t a = s_u32(b);
    uint32_t done = 0;
    long long t0 = 0;
    for (int spin = 0; !done; ++spin) {
        asm volatile("{\n\t.reg .pred p;\n\tmbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\tselp.u32 %0, 1, 0, p;\n\t}" : "=r"(done) : "r"(a), "r"(parity) : "memory");
        if (!done) {
            if (SLEEP) __nanosleep(spin < 4 ? 40 : 200);
            if (spin > 256) {       // a barrier that never completes is a bug: trap instead of hanging the device
                if (t0 == 0) t0 = clock64();
                else if (clock64() - t0 > (1ll << 31)) __trap();
            }
        }
    }
}
#ifdef PDP_NN_TIMING
__device__ long long g_nn_log[96][8];       // CTA 0, first 96 chunks: 0 producer sees empty, 1 producer arrives, 2 B copy issued, 3 issuer sees full, 4 MMAs issued, 5 commit done
#define NN_LOG(chunk_, ev_) do { if (blockIdx.x == 0 && (chunk_) < 96) g_nn_log[chunk_][ev_] = clock64(); } while (0)
__device__ long long g_nn_plog[96][32];     // CTA 0, first 96 chunks, producer warp w: [w] data in registers, [8 + w] empty seen, [16 + w] arrived
#define NN_PLOG(chunk_, ev_) do { if (blockIdx.x == 0 && (chunk_) < 96 && lane == 0) g_nn_plog[chunk_][8 * (ev_) + warp] = clock64(); } while (0)
__device__ unsigned long long g_nn_wait[8];     // cycles waited: 0 A-prod on empty, 1 B-prod on empty, 2 issuer on full_a, 3 on full_b, 4 on acc_empty, 5 epilogue on acc_full, 6 issuer total, 7 epilogue busy
#define MB_WAIT_T(bar, par, slot) do { const long long _t0 = clock64(); mb_wait<((slot) < 2 || (slot) > 4)>(bar, par); if ((threadIdx.x & 31) == 0) atomicAdd(&g_nn_wait[slot], (unsigned long long)(clock64() - _t0)); } while (0)
#else
#define MB_WAIT_T(bar, par, slot) mb_wait<((slot) < 2 || (slot) > 4)>(bar, par)     // slots 2-4: the MMA issuer polls without backing off
#define NN_LOG(chunk_, ev_) do {} while (0)
#define NN_PLOG(chunk_, ev_) do {} while (0)
#endif
__device__ __forceinline__ void bulk_load(void* dst, const void* src, uint32_t bytes, uint64_t* bar) {
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(s_u32(dst)), "l"(src), "r"(bytes), "r"(s_u32(bar)) : "memory");
}
// one lane of the (converged) warp
__device__ __forceinline__ bool elect_one() {
    uint32_t pred;
    asm volatile("{\n\t.reg .pred p;\n\telect.sync _|p, 0xffffffff;\n\tselp.u32 %0, 1, 0, p;\n\t}" : "=r"(pred));
    return pred != 0u;
}
__device__ __forceinline__ void fence_async_smem() { asm volatile("fence.proxy.async.shared::cta;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_after() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_commit(uint64_t* b) { asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(s_u32(b)) : "memory"); }
// D[tmem] (+)= A[smem] B[smem]^T, tf32 inputs, fp32 accumulation
__device__ __forceinline__ void tc_mma_tf32(uint32_t tmem_d, uint64_t desc_a, uint64_t desc_b, uint32_t idesc, uint32_t accumulate) {
    asm volatile("{\n\t.reg .pred p;\n\tsetp.ne.b32 p, %4, 0;\n\ttcgen05.mma.cta_group::1.kind::tf32 [%0], %1, %2, %3, p;\n\t}"
                 ::"r"(tmem_d), "l"(desc_a), "l"(desc_b), "r"(idesc), "r"(accumulate) : "memory");
}
// shared-memory matrix descriptor, K-major, no swizzle: start address, LBO (next 16-byte column group), SBO (next 8 rows)
__device__ __forceinline__ uint64_t smem_desc(uint32_t addr, uint32_t lbo_bytes, uint32_t sbo_bytes, uint32_t layout_type = 0) {
    return (uint64_t)((addr >> 4) & 0x3fffu) | ((uint64_t)((lbo_bytes >> 4) & 0x3fffu) << 16) | ((uint64_t)((sbo_bytes >> 4) & 0x3fffu) << 32) |
           ((uint64_t)1 << 46) |    // descriptor version of sm_100
           ((uint64_t)(layout_type & 7u) << 61);   // 0 no swizzle, 2 128-byte, 4 64-byte, 6 32-byte swizzle
}
// instruction descriptor of kind::tf32: D fp32, A and B tf32, both K-major, N >> 3 at bit 17, M >> 4 at bit 24
__device__ __forceinline__ uint32_t instr_desc(int m, int n) {
    return (1u << 4) | (2u << 7) | (2u << 10) | ((uint32_t)(n >> 3) << 17) | ((uint32_t)(m >> 4) << 24);
}
// 16 consecutive accumulator columns of this thread's lane
__device__ __forceinline__ void tc_ld16(uint32_t taddr, float (&v)[16]) {
    uint32_t r[16];
    asm volatile("tcgen05.ld.sync.aligned.32x32b.x16.b32 {%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15}, [%16];"
                 : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]), "=r"(r[8]), "=r"(r[9]),
                   "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15])
                 : "r"(taddr));
    asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
#pragma unroll
    for (int i = 0; i < 16; ++i) v[i] = __uint_as_float(r[i]);
}

// Epilogue activations on the special-function unit (ex2 / lg2 / rcp: relative error ~1e-6 on O(1) arguments, an order
// below the three-term product's own error); the IEEE forms cost the epilogue warps four times the issue slots, and the
// epilogue shares the SM's schedulers with the operand staging.
__device__ __forceinline__ float logsigmoidf(float x) { return fminf(x, 0.f) - __logf(1.f + __expf(-fabsf(x))); }   // F.logsigmoid
__device__ __forceinline__ float sigmoidf_(float x) { return __fdividef(1.f, 1.f + __expf(-x)); }
__device__ __forceinline__ float tanhf_(float x) { return 2.f * sigmoidf_(2.f * x) - 1.f; }

// element k of the concatenated row
__device__ __forceinline__ float a_elem(const EdgeNNArgs& P, int64_t row, int k) {
    if (k < P.ks[0]) return __ldg(P.src[0] + row * P.ks[0] + k);
    k -= P.ks[0];
    if (k < P.ks[1]) return __ldg(P.src[1] + row * P.ks[1] + k);
    k -= P.ks[1];
    if (k < P.ks[2]) return __ldg(P.src[2] + row * P.ks[2] + k);
    return 0.f;
}

template <int EPI>
__global__ void __launch_bounds__(kThreads, 1) k_edge_nn(const __grid_constant__ EdgeNNArgs P) {
    extern __shared__ __align__(1024) unsigned char smem[];
    __shared__ __align__(8) uint64_t bar_full[4], bar_empty[4], bar_acc_full[2], bar_acc_empty[2], bar_ovl[2];
    __shared__ uint32_t tmem_base_s;
    __shared__ uint32_t issue_turn;                  // number of the chunk whose MMAs may be issued next
    __shared__ int2 s_cd[2][kMaxChunks];             // per half chunk: {source (-1: element by element), column in it}
    __shared__ __align__(16) float s_bias[768];                   // the layer's (padded) bias: passes * n_tot values
    const int tid = threadIdx.x, lane = tid & 31;
    const int warp = __shfl_sync(0xffffffffu, tid >> 5, 0);      // (a broadcast: the compiler treats the role dispatch as warp-uniform)
    const int S = P.stages;
    const uint32_t a_bytes = 2u * kTileM * kChunkK * 4u;                 // hi + lo
    const uint32_t b_bytes = 2u * (uint32_t)P.n_tot * kChunkK * 4u;
    const uint32_t stage_bytes = a_bytes + b_bytes;
    for (int i = tid; i < P.passes * P.n_tot; i += kThreads) s_bias[i] = __ldg(P.bias + i);
    for (int i = tid; i < 2 * P.k_chunks; i += kThreads) {
        const int c = i >> 1, hf = i & 1;
        int k = c * kChunkK + kHalfK * hf, si = 0;
        while (si < 2 && k >= P.ks[si]) { k -= P.ks[si]; ++si; }
        const bool copy = k + kHalfK <= P.ks[si] && !((k | P.ks[si]) & 1) && !((uintptr_t)P.src[si] & 7);
        s_cd[hf][c] = make_int2(copy ? si : -1, k);
    }
    if (tid == 0) {
        issue_turn = 0u;
        for (int s = 0; s < S; ++s) { mb_init(&bar_full[s], 9); mb_init(&bar_empty[s], 1); }     // full: 8 A-producer warps + the weight copy (arrive + bytes)
        for (int b = 0; b < 2; ++b) { mb_init(&bar_acc_full[b], 1); mb_init(&bar_acc_empty[b], 8); mb_init(&bar_ovl[b], 8); }
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    if (warp == 16) {    // the accumulators: all 512 columns of tensor memory (one CTA per SM)
        asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], 512;" ::"r"(s_u32(&tmem_base_s)) : "memory");
        asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
    }
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem_base = tmem_base_s;

    const int64_t n_tiles = (P.rows + kTileM - 1) / kTileM;
    const int units = P.passes * P.k_chunks;       // chunk iterations per tile
    // accumulator buffers: columns [0, n_tot) and [buf1, buf1 + n_tot); they share n_ovl columns when a pass is wider than 256
    const uint32_t buf1 = P.n_tot > 256 ? (uint32_t)(512 - P.n_tot) : 256u;
    const int n_ovl = P.n_tot > 256 ? 2 * P.n_tot - 512 : 0;
    // every role walks the same sequence of (tile, pass, chunk) and keeps its own ring position
    if (warp < 8) {
        // ---------------- A producers: threads r and r + 128 <-> row r of the tile, column groups {0,1} / {2,3} of the chunk.
        // A thread's 32 bytes of a chunk travel global -> shared memory as four 8-byte asynchronous copies (cp.async) into a
        // ring of thread-private slots, kRawDepth chunks ahead, and are picked up with cp.async.wait_group: no register is
        // held for data in flight, and the oldest group is the only one waited for.  (With the prefetched chunks in
        // registers the unrolled ring shared scoreboards between its stages: every fourth chunk waited for the youngest
        // loads, 1 000 - 2 700 cycles, and the address arithmetic of the loads took 480 cycles per chunk, both measured with
        // the -DPDP_NN_TIMING build.)  Where the 8 columns come from is looked up per chunk in a table built at kernel start:
        // one source at an even offset with rows of even length -> copies; anything else (a span across two sources, an odd
        // offset, rows of odd length) element by element through registers.
        const int r = tid & 127, half = tid >> 7;
        int s = 0; uint32_t ph = 0;
        const int64_t tile_step = (int64_t)gridDim.x * kTileM;
        const int64_t my_tiles = (n_tiles - blockIdx.x + gridDim.x - 1) / gridDim.x;
        const int64_t total = my_tiles * units;
        // ring level l: two 16-byte slots per thread, slot A of thread t at + 8192 l + 16 t, slot B 4096 further
        const uint32_t raw_sa = s_u32(smem + (size_t)S * stage_bytes) + 16u * (uint32_t)tid;
        int64_t pf_row = (int64_t)blockIdx.x * kTileM + r;      // prefetch cursor: row of this thread, chunk of the pass, pass
        int pf_c = 0, pf_p = 0;
        const float *rp0 = nullptr, *rp1 = nullptr, *rp2 = nullptr;      // this thread's row in the three sources
        auto row_ptrs = [&]() {
            rp0 = P.src[0] + pf_row * P.ks[0];
            rp1 = P.ks[1] ? P.src[1] + pf_row * P.ks[1] : nullptr;
            rp2 = P.ks[2] ? P.src[2] + pf_row * P.ks[2] : nullptr;
        };
        row_ptrs();
        // The thread's 32 bytes are 8-byte aligned.  Where they are 16-byte aligned they go as two 16-byte copies (slot A, slot
        // B); where not -- every other row of a 600-byte-row tensor -- the aligned middle goes as one 16-byte copy (slot A)
        // and the two ends as 8-byte copies (the halves of slot B): 2.5 copies per thread and chunk instead of four of 8 bytes
        // (what the layers wait for is the L1 tag stage taking the threads' sectors one by one).
        auto fetch = [&](int level) {
            if (pf_row < P.rows) {
                const int2 e = s_cd[half][pf_c];
                const uint32_t dst = raw_sa + 8192u * (uint32_t)level;
                if (e.x >= 0) {
                    const float* p = (e.x == 0 ? rp0 : (e.x == 1 ? rp1 : rp2)) + e.y;
                    if (!((uintptr_t)p & 8)) {
                        asm volatile("cp.async.ca.shared.global [%0], [%1], 16;" ::"r"(dst), "l"(p) : "memory");
                        asm volatile("cp.async.ca.shared.global [%0], [%1], 16;" ::"r"(dst + 4096u), "l"(p + 4) : "memory");
                    } else {
                        asm volatile("cp.async.ca.shared.global [%0], [%1], 16;" ::"r"(dst), "l"(p + 2) : "memory");
                        asm volatile("cp.async.ca.shared.global [%0], [%1], 8;" ::"r"(dst + 4096u), "l"(p) : "memory");
                        asm volatile("cp.async.ca.shared.global [%0], [%1], 8;" ::"r"(dst + 4104u), "l"(p + 6) : "memory");
                    }
                } else {
                    const int k0 = pf_c * kChunkK + kHalfK * half;
                    float x[kHalfK];
#pragma unroll
                    for (int j = 0; j < kHalfK; ++j) x[j] = a_elem(P, pf_row, k0 + j);
                    asm volatile("st.shared.v4.f32 [%0], {%1, %2, %3, %4};" ::"r"(dst), "f"(x[0]), "f"(x[1]), "f"(x[2]), "f"(x[3]) : "memory");
                    asm volatile("st.shared.v4.f32 [%0], {%1, %2, %3, %4};" ::"r"(dst + 4096u), "f"(x[4]), "f"(x[5]), "f"(x[6]), "f"(x[7]) : "memory");
                }
            }
            asm volatile("cp.async.commit_group;" ::: "memory");
            if (++pf_c == P.k_chunks) {
                pf_c = 0;
                if (++pf_p == P.passes) { pf_p = 0; pf_row += tile_step; row_ptrs(); }
            }
        };
        for (int d = 0; d < kRawDepth; ++d) fetch(d);        // (groups past the end are empty: the count stays uniform)
        int64_t c_row = (int64_t)blockIdx.x * kTileM + r;        // consumer cursor: row, unit of the tile, chunk of the pass
        int c_u = 0, c_c = 0, level = 0;
        // bit 3 of the address of this thread's row in each source (the consumer re-derives which form the copies took)
        uint32_t par0 = 0, par1 = 0, par2 = 0;
        auto row_parity = [&]() {
            par0 = (uint32_t)(((uintptr_t)(P.src[0] + c_row * P.ks[0]) >> 3) & 1);
            par1 = P.ks[1] ? (uint32_t)(((uintptr_t)(P.src[1] + c_row * P.ks[1]) >> 3) & 1) : 0u;
            par2 = P.ks[2] ? (uint32_t)(((uintptr_t)(P.src[2] + c_row * P.ks[2]) >> 3) & 1) : 0u;
        };
        row_parity();
        // rows of 64 bytes, the 16-byte unit g of row r at unit g ^ ((r >> 1) & 3): Swizzle<2,4,3>
        const uint32_t off0 = (uint32_t)(r * 64 + (((2 * half) ^ ((r >> 1) & 3)) << 4)), off1 = (uint32_t)(r * 64 + (((2 * half + 1) ^ ((r >> 1) & 3)) << 4));
        for (int64_t g0 = 0; g0 < total; ++g0) {
            const bool live = c_row < P.rows;
            asm volatile("cp.async.wait_group %0;" ::"n"(kRawDepth - 1) : "memory");
            float v[kHalfK];
            {
                const uint32_t src = raw_sa + 8192u * (uint32_t)level;
                float a[4], bq[4];
                asm volatile("ld.shared.v4.f32 {%0, %1, %2, %3}, [%4];" : "=f"(a[0]), "=f"(a[1]), "=f"(a[2]), "=f"(a[3]) : "r"(src) : "memory");
                asm volatile("ld.shared.v4.f32 {%0, %1, %2, %3}, [%4];" : "=f"(bq[0]), "=f"(bq[1]), "=f"(bq[2]), "=f"(bq[3]) : "r"(src + 4096u) : "memory");
                const int2 e = s_cd[half][c_c];
                const bool sh = e.x >= 0 && ((((e.x == 0 ? par0 : (e.x == 1 ? par1 : par2)) + ((uint32_t)e.y >> 1)) & 1u) != 0u);
                v[0] = sh ? bq[0] : a[0]; v[1] = sh ? bq[1] : a[1];
                v[2] = sh ? a[0] : a[2];  v[3] = sh ? a[1] : a[3];
                v[4] = sh ? a[2] : bq[0]; v[5] = sh ? a[3] : bq[1];
                v[6] = bq[2]; v[7] = bq[3];
            }
            uint4 hi[2], lo[2];
#pragma unroll
            for (int gg = 0; gg < 2; ++gg) {
                uint32_t* hp = reinterpret_cast<uint32_t*>(&hi[gg]);
                uint32_t* lp = reinterpret_cast<uint32_t*>(&lo[gg]);
#pragma unroll
                for (int j = 0; j < 4; ++j) {
                    const float x = live ? v[4 * gg + j] : 0.f;
                    const uint32_t hb = __float_as_uint(x) & 0xffffe000u;
                    hp[j] = hb;
                    lp[j] = __float_as_uint(x - __uint_as_float(hb)) & 0xffffe000u;
                }
            }
            NN_PLOG((int)g0, 3);
            fetch(level);                                        // the slot just read takes the chunk kRawDepth further on
            if (++level == kRawDepth) level = 0;
            NN_PLOG((int)g0, 0);
            MB_WAIT_T(&bar_empty[s], ph ^ 1u, 0);
            NN_PLOG((int)g0, 1);
            if (tid == 0) NN_LOG((int)g0, 0);
            unsigned char* st = smem + (size_t)s * stage_bytes;
            *reinterpret_cast<uint4*>(st + off0) = hi[0];
            *reinterpret_cast<uint4*>(st + off1) = hi[1];
            *reinterpret_cast<uint4*>(st + (size_t)(kTileM * kChunkK * 4) + off0) = lo[0];
            *reinterpret_cast<uint4*>(st + (size_t)(kTileM * kChunkK * 4) + off1) = lo[1];
            fence_async_smem();          // these generic-proxy writes are read by the tensor core (async proxy)
            __syncwarp();
            if (lane == 0) mb_arrive(&bar_full[s]);      // one arrival per warp: 256 arrivals on one barrier word serialise
            NN_PLOG((int)g0, 2);
            if (tid == 0) NN_LOG((int)g0, 1);
            if (++s == S) { s = 0; ph ^= 1u; }
            if (++c_c == P.k_chunks) c_c = 0;
            if (++c_u == units) { c_u = 0; c_row += tile_step; row_parity(); }
        }
        asm volatile("cp.async.wait_group 0;" ::: "memory");
    } else if (warp == 17 && lane == 0) {
        // ---------------- B producer: one bulk copy per chunk
        int s = 0; uint32_t ph = 0;
        int gb = 0;
        for (int64_t tile = blockIdx.x; tile < n_tiles; tile += gridDim.x) {
            for (int u = 0; u < units; ++u, ++gb) {
                MB_WAIT_T(&bar_empty[s], ph ^ 1u, 1);
                NN_LOG(gb, 2);
                mb_expect_tx(&bar_full[s], b_bytes);
                bulk_load(smem + (size_t)s * stage_bytes + a_bytes, reinterpret_cast<const unsigned char*>(P.w_img) + (size_t)u * b_bytes, b_bytes, &bar_full[s]);
                if (++s == S) { s = 0; ph ^= 1u; }
            }
        }
    } else if (warp == 16 || warp == 18) {
        // ---------------- MMA issuers: two warps take the chunks in turn.  The whole warp walks the loop so that descriptors
        //                  and addresses are warp-uniform values (uniform registers: a lone thread's per-thread values cost
        //                  five R2UR moves per MMA, 150-180 cycles of issue time each); one elected lane issues.  Around a
        //                  chunk's MMAs a warp waits for the stage, fences and commits: with two warps one's bookkeeping runs
        //                  under the other's MMAs.  The MMAs of a pass accumulate into one buffer and must be issued in chunk
        //                  order: a turn counter in shared memory hands the pipe from one warp to the other (commit tracks the
        //                  issuing thread's own MMAs; the pipe runs in issue order, so the last chunk's completion implies
        //                  the whole pass).
        const int me = (warp == 16) ? 0 : 1;
        const int w0 = P.n_tot < kMmaN ? P.n_tot : kMmaN, w1 = P.n_tot - w0;      // columns of the two MMAs of a k-step and term
        const uint32_t idesc0 = instr_desc(kTileM, w0), idesc1 = instr_desc(kTileM, w1 > 0 ? w1 : 16);
        // K-major, 64-byte swizzle: rows of 64 bytes, 8-row atoms of 512 bytes one after the other (SBO = 512); a k-step of 8
        // elements = 32 bytes further along the row (the hardware applies the XOR to the address it computes)
        const uint64_t desc_hi_a = smem_desc(0, 16, 512, 4), desc_hi_b = smem_desc(0, 16, 512, 4);
        const uint32_t kstep4 = 32u >> 4, nrow4 = 64u >> 4;
        const uint32_t smem_a4 = s_u32(smem) >> 4, stage4 = stage_bytes >> 4;
        const uint32_t a_lo4 = (kTileM * kChunkK * 4) >> 4, b_off4 = a_bytes >> 4, b_lo4 = ((uint32_t)P.n_tot * kChunkK * 4) >> 4;
        int s = 0; uint32_t ph = 0, acc_ph0 = 0u, acc_ph1 = 0u, ovl_ph0 = 0u, ovl_ph1 = 0u;
        int ab = 0;                                     // accumulator buffer of this pass
        uint32_t g = 0;                                 // running chunk number
        bool first_pass = true;
        volatile uint32_t* turn = &issue_turn;
        for (int64_t tile = blockIdx.x; tile < n_tiles; tile += gridDim.x) {
            for (int p = 0; p < P.passes; ++p) {
                const uint32_t tacc = tmem_base + (ab ? buf1 : 0u);
                for (int c = 0; c < P.k_chunks; ++c, ++g) {
                    if ((int)(g & 1u) == me) {
                        if (c == 0) {
                            MB_WAIT_T(&bar_acc_empty[ab], (ab ? acc_ph1 : acc_ph0) ^ 1u, 4);   // the epilogue has read this buffer's previous contents
                            // ... and, of the pass before this one (the other buffer), the columns the two buffers share
                            if (n_ovl > 0 && !first_pass) MB_WAIT_T(&bar_ovl[ab ^ 1], ab ? ovl_ph0 : ovl_ph1, 4);
                        }
                        MB_WAIT_T(&bar_full[s], ph, 2);
                        NN_LOG((int)g, 3);
                        while (*turn != g) { }              // the other warp has issued chunk g - 1
                        tc_fence_after();
                        // descriptors = constant upper parts | (address >> 4): everything below is 32-bit adds on the low word
                        const uint32_t sa4 = (smem_a4 + (uint32_t)s * stage4);
                        const bool leader = elect_one();
#pragma unroll
                        for (int ks = 0; ks < kChunkK / 8; ++ks) {
#pragma unroll
                            for (int term = 0; term < 3; ++term) {      // hi hi, lo hi, hi lo
                                const uint32_t a4 = sa4 + (term == 1 ? a_lo4 : 0u) + ks * kstep4;
                                const uint32_t b4 = sa4 + b_off4 + (term == 2 ? b_lo4 : 0u) + ks * kstep4;
                                const uint32_t nb4 = (uint32_t)w0 * nrow4;
                                const uint32_t acc = (c == 0 && ks == 0 && term == 0) ? 0u : 1u;
                                if (leader) {
                                    tc_mma_tf32(tacc, desc_hi_a | a4, desc_hi_b | b4, idesc0, acc);
                                    if (w1 > 0) tc_mma_tf32(tacc + (uint32_t)w0, desc_hi_a | a4, desc_hi_b | (b4 + nb4), idesc1, acc);
                                }
                            }
                        }
                        NN_LOG((int)g, 4);
                        if (leader) {
                            __threadfence_block();
                            *turn = g + 1;                       // hand the pipe over
                            tc_commit(&bar_empty[s]);            // the stage is free once these MMAs have read it
                            if (c == P.k_chunks - 1) tc_commit(&bar_acc_full[ab]);
                        }
                        __syncwarp();
                        NN_LOG((int)g, 5);
                    }
                    if (++s == S) { s = 0; ph ^= 1u; }
                }
                if (ab) acc_ph1 ^= 1u; else acc_ph0 ^= 1u;
                if (n_ovl > 0 && !first_pass) { if (ab) ovl_ph0 ^= 1u; else ovl_ph1 ^= 1u; }      // (the other buffer's barrier was waited for)
                first_pass = false;
                ab ^= 1;
            }
        }
    }
    if (warp >= 8 && warp < 16) {
        // ---------------- epilogue: thread <-> accumulator lane = row of the tile; two warps per lane quadrant, each takes
        //                  every other group of 16 columns.  A thread's 16 results are contiguous in its output row: 64-bit
        //                  accesses (rows are 8-byte aligned when their length is even and the array starts 8-byte aligned),
        //                  two full sectors per thread.  The caller's arrays need only be 4-byte aligned: a view that starts
        //                  one float into its storage takes the element-by-element path.  (h_old is null for LINEAR.)
        const int q = warp & 3;                      // lane quadrant this warp may read (warp index mod 4)
        const int hh = (warp - 8) >> 2;              // which half of the column groups
        const int r = q * 32 + lane;
        const uint32_t tlane0 = tmem_base + ((uint32_t)(q * 32) << 16);
        const bool vec2 = !(P.n_out & 1) && !(((uintptr_t)P.out | (uintptr_t)P.h_old) & 7);
        uint32_t acc_ph[2] = {0u, 0u};
        int ab = 0;
        // LINEAR: a tile's output rows are consecutive in global memory, so the warps collect them in a shared-memory image of
        // the tile and one thread sends it off with ONE bulk store (cp.async.bulk.global.shared).  Thread-per-row stores touch
        // 32 sectors per warp instruction and the L1 tag stage takes them one by one: with the row-strided operand loads
        // they were what the layer was bound by (0.66 -> 0.48 ms for 151 -> 100 over 1.2 M rows).  The GRU cell's tile (77 KB)
        // only fits beside its stages with a shorter copy ring and no L1 to speak of: measured 3.1 ms against 2.6 ms, not done.
        const bool otile_on = EPI == EPI_LINEAR && P.out_tile != 0;
        float* otile = reinterpret_cast<float*>(smem + (size_t)S * stage_bytes + kRawBytes);
        auto store16 = [&](float* dst, const float (&y)[16], int nvalid) {      // nvalid of the 16 values exist
            if (vec2 && nvalid == 16) {
                if (!((uintptr_t)dst & 15)) {
#pragma unroll
                    for (int j = 0; j < 4; ++j) reinterpret_cast<float4*>(dst)[j] = make_float4(y[4 * j], y[4 * j + 1], y[4 * j + 2], y[4 * j + 3]);
                } else {
#pragma unroll
                    for (int j = 0; j < 8; ++j) reinterpret_cast<float2*>(dst)[j] = make_float2(y[2 * j], y[2 * j + 1]);
                }
            } else {
#pragma unroll
                for (int j = 0; j < 16; ++j) if (j < nvalid) dst[j] = y[j];
            }
        };
        for (int64_t tile = blockIdx.x; tile < n_tiles; tile += gridDim.x) {
            const int64_t row = tile * kTileM + r;
            const bool live = row < P.rows;
            const float mk = (live && P.row_mask) ? __ldg(P.row_mask + row) : 1.f;
            if (otile_on) {      // the previous tile's bulk store has read the image
                if (tid == 256) asm volatile("cp.async.bulk.wait_group.read 0;" ::: "memory");
                asm volatile("bar.sync 2, 256;" ::: "memory");
            }
            for (int p = 0; p < P.passes; ++p) {
                MB_WAIT_T(&bar_acc_full[ab], acc_ph[ab], 5);
                acc_ph[ab] ^= 1u;
                tc_fence_after();
                const uint32_t tlane = tlane0 + (ab ? buf1 : 0u);
                if (EPI == EPI_LINEAR) {
                    for (int c0 = 16 * hh; c0 < P.n_tot; c0 += 32) {
                        float v[16];
                        tc_ld16(tlane + (uint32_t)c0, v);
                        const int n0 = p * P.n_tot + c0;
                        if (!live || n0 >= P.n_out) continue;
                        float y[16], bq[16];
#pragma unroll
                        for (int j = 0; j < 4; ++j) {      // (n0 is a multiple of 16: 64-byte aligned)
                            const float4 b4 = reinterpret_cast<const float4*>(s_bias + n0)[j];
                            bq[4 * j] = b4.x; bq[4 * j + 1] = b4.y; bq[4 * j + 2] = b4.z; bq[4 * j + 3] = b4.w;
                        }
#pragma unroll
                        for (int j = 0; j < 16; ++j) {
                            float t = v[j] + bq[j];
                            if (P.act == ACT_LOGSIGMOID) t = logsigmoidf(t);
                            if (P.row_mask) t *= mk;
                            y[j] = t;
                        }
                        store16(otile_on ? otile + (size_t)r * P.n_out + n0 : P.out + row * P.n_out + n0, y, min(16, P.n_out - n0));
                    }
                } else {
                    // the pass holds hidden units [p * nh, (p + 1) * nh), four columns each: r, z, W_in x, W_hn h of the unit.  A
                    // group of 16 columns = four whole units.  The columns this buffer shares with the other one go first (of
                    // buffer 0 its last n_ovl columns, of buffer 1 its first): once every warp has read its part of them, the
                    // MMAs of the next pass -- into the other buffer -- may start, under the rest of this epilogue.
                    const int nh = P.n_tot / 4, ngrp = P.n_tot / 16, novl = n_ovl / 16;
                    const int g_first = ab ? 0 : ngrp - novl;
                    const float* bs = s_bias + (size_t)p * P.n_tot;
                    bool handed = novl == 0;
                    for (int i = hh; i < ngrp; i += 2) {
                        if (!handed && i >= novl) {
                            tc_fence_before();
                            __syncwarp();
                            if (lane == 0) mb_arrive(&bar_ovl[ab]);
                            handed = true;
                        }
                        int grp = i + g_first;
                        if (grp >= ngrp) grp -= ngrp;
                        float v[16];
                        tc_ld16(tlane + (uint32_t)(16 * grp), v);
                        const int u0 = p * nh + 4 * grp;
                        if (!live || u0 >= P.n_out) continue;
                        const int nvalid = min(4, P.n_out - u0);
                        float ho[4], y[4];
                        const float* hp = P.h_old + row * P.n_out + u0;
                        if (vec2 && nvalid == 4) {       // 16-byte aligned in every other row of a 600-byte-row tensor: one access, else two
                            if (!((uintptr_t)hp & 15)) {
                                const float4 t4 = __ldg(reinterpret_cast<const float4*>(hp));
                                ho[0] = t4.x; ho[1] = t4.y; ho[2] = t4.z; ho[3] = t4.w;
                            } else {
#pragma unroll
                                for (int j = 0; j < 2; ++j) { const float2 t2 = __ldg(reinterpret_cast<const float2*>(hp) + j); ho[2 * j] = t2.x; ho[2 * j + 1] = t2.y; }
                            }
                        } else {
#pragma unroll
                            for (int j = 0; j < 4; ++j) ho[j] = j < nvalid ? __ldg(hp + j) : 0.f;
                        }
                        const float4* bg = reinterpret_cast<const float4*>(bs + 16 * grp);      // (n_tot is a multiple of 16: 64-byte aligned)
#pragma unroll
                        for (int j = 0; j < 4; ++j) {
                            const float4 b4 = bg[j];
                            const float rg = sigmoidf_(v[4 * j] + b4.x);
                            const float zg = sigmoidf_(v[4 * j + 1] + b4.y);
                            const float ng = tanhf_(v[4 * j + 2] + b4.z + rg * (v[4 * j + 3] + b4.w));
                            float hn = (1.f - zg) * ng + zg * ho[j];
                            if (P.row_mask) hn = mk * hn + (1.f - mk) * ho[j];
                            y[j] = hn;
                        }
                        float* dst = P.out + row * P.n_out + u0;
                        if (vec2 && nvalid == 4) {
                            if (!((uintptr_t)dst & 15)) {
                                *reinterpret_cast<float4*>(dst) = make_float4(y[0], y[1], y[2], y[3]);
                            } else {
                                reinterpret_cast<float2*>(dst)[0] = make_float2(y[0], y[1]);
                                reinterpret_cast<float2*>(dst)[1] = make_float2(y[2], y[3]);
                            }
                        } else {
#pragma unroll
                            for (int j = 0; j < 4; ++j) if (j < nvalid) dst[j] = y[j];
                        }
                    }
                    if (!handed) {
                        tc_fence_before();
                        __syncwarp();
                        if (lane == 0) mb_arrive(&bar_ovl[ab]);
                    }
                }
                tc_fence_before();
                __syncwarp();
                if (lane == 0) mb_arrive(&bar_acc_empty[ab]);
                ab ^= 1;
            }
            if (otile_on) {
                fence_async_smem();                                  // the image was written through the generic proxy
                asm volatile("bar.sync 2, 256;" ::: "memory");
                if (tid == 256) {
                    const int64_t row0 = tile * kTileM;
                    const int64_t nrow = (P.rows - row0 < kTileM) ? (P.rows - row0) : kTileM;
                    const uint32_t bytes = (uint32_t)(nrow * P.n_out * 4), b16 = bytes & ~15u;
                    float* gdst = P.out + row0 * P.n_out;
                    if (b16) asm volatile("cp.async.bulk.global.shared::cta.bulk_group [%0], [%1], %2;" ::"l"(gdst), "r"(s_u32(otile)), "r"(b16) : "memory");
                    asm volatile("cp.async.bulk.commit_group;" ::: "memory");
                    for (uint32_t i = b16 / 4; i < bytes / 4; ++i) gdst[i] = otile[i];      // (a last tile whose bytes are no multiple of 16)
                }
            }
        }
        if (otile_on && tid == 256) asm volatile("cp.async.bulk.wait_group 0;" ::: "memory");
    }
    tc_fence_before();
    __syncthreads();
    if (warp == 16) {
        tc_fence_after();
        asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, 512;" ::"r"(tmem_base) : "memory");
    }
}

int launch(EdgeNNArgs& P, int epi, cudaStream_t stream) {
    int dev = 0, sms = 0, cc = 0;
    if (cudaGetDevice(&dev) != cudaSuccess || cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev) != cudaSuccess ||
        cudaDeviceGetAttribute(&cc, cudaDevAttrComputeCapabilityMajor, dev) != cudaSuccess) { pdp_set_error("pdp_edge_nn: no CUDA device"); return PDP_ERR_CUDA; }
    if (cc < 10) { pdp_set_error("pdp_edge_nn: tcgen05 needs sm_100a"); return PDP_ERR_UNSUPPORTED; }
    const size_t stage = 2u * kTileM * kChunkK * 4u + 2u * (size_t)P.n_tot * kChunkK * 4u;
    const size_t smem = stage * P.stages + kRawBytes + (P.out_tile ? (size_t)kTileM * P.n_out * 4 : 0);
    void* kern = epi == EPI_GRU ? (void*)k_edge_nn<EPI_GRU> : (void*)k_edge_nn<EPI_LINEAR>;
    cudaError_t e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (e != cudaSuccess) { pdp_set_error("pdp_edge_nn: shared memory %zu: %s", smem, cudaGetErrorString(e)); return PDP_ERR_CUDA; }
    const int64_t n_tiles = (P.rows + kTileM - 1) / kTileM;
    const int grid = (int)(n_tiles < sms ? n_tiles : sms);
    if (epi == EPI_GRU) k_edge_nn<EPI_GRU><<<grid, kThreads, smem, stream>>>(P);
    else k_edge_nn<EPI_LINEAR><<<grid, kThreads, smem, stream>>>(P);
    e = cudaGetLastError();
    if (e != cudaSuccess) { pdp_set_error("pdp_edge_nn: launch -> %s", cudaGetErrorString(e)); return PDP_ERR_CUDA; }
    return PDP_OK;
}

bool fill_common(EdgeNNArgs& P, const float* x1, int k1, const float* x2, int k2, const float* x3, int k3, int64_t rows, const float* w_img,
                 const float* bias, int n_blk, int n_mma, int passes, const char* who) {
    P.src[0] = x1; P.src[1] = x2; P.src[2] = x3;
    P.ks[0] = k1 > 0 ? k1 : 0; P.ks[1] = k2 > 0 ? k2 : 0; P.ks[2] = k3 > 0 ? k3 : 0;
    P.k_total = P.ks[0] + P.ks[1] + P.ks[2];
    P.k_chunks = (P.k_total + kChunkK - 1) / kChunkK;
    P.rows = rows; P.w_img = w_img; P.bias = bias;
    P.n_blk = n_blk; P.n_mma = n_mma; P.n_tot = n_blk * n_mma; P.passes = passes;
    if (P.k_total <= 0 || !w_img || !bias || n_blk < 16 || (n_blk & 15) || n_mma < 1 || P.n_tot > kMaxNTot || passes < 1 ||
        (k1 > 0 && !x1) || (k2 > 0 && !x2) || (k3 > 0 && !x3) || ((uintptr_t)w_img & 15) || passes * n_blk * n_mma > 768 || P.k_chunks > kMaxChunks) {
        pdp_set_error("%s: bad argument (k=%d n_blk=%d n_mma=%d passes=%d)", who, P.k_total, n_blk, n_mma, passes);
        return false;
    }
    const size_t stage = 2u * kTileM * kChunkK * 4u + 2u * (size_t)P.n_tot * kChunkK * 4u;
    // Few stages on purpose: what the ring does not take stays L1, and the row-strided reads of the operand staging and of the
    // epilogue live on L1 hits (GRU cell over 1.2 M rows: 4 stages 4.14 ms, 3 stages 3.61 ms, 2 stages 3.50 ms)
    int st = (int)((100 * 1024) / stage);
    P.stages = st > 4 ? 4 : (st < 2 ? 2 : st);
    if (const char* e = getenv("PDP_B200_NN_STAGES")) { const int v = atoi(e); if (v >= 2 && v <= 4 && (size_t)v * stage + kRawBytes <= 220 * 1024) P.stages = v; }   // (profiling)
    return true;
}

}  // namespace

// One dense layer over rows: out[rows, n_out] = act([x1 | x2 | x3] W^T + bias) (* row_mask).  w_img / bias: the tiled
// weight image and padded bias built by pdp_solver_b200/nn/tensor_ops.py (n_blk columns per MMA, n_mma blocks per pass).
#ifdef PDP_NN_TIMING
extern "C" int pdp_edge_nn_event_log(long long* host_96x8) {
    return cudaMemcpyFromSymbol(host_96x8, g_nn_log, sizeof(long long) * 96 * 8) == cudaSuccess ? PDP_OK : PDP_ERR_CUDA;
}
extern "C" int pdp_edge_nn_producer_log(long long* host_96x24) {
    return cudaMemcpyFromSymbol(host_96x24, g_nn_plog, sizeof(long long) * 96 * 32) == cudaSuccess ? PDP_OK : PDP_ERR_CUDA;
}
extern "C" int pdp_edge_nn_wait_counters(unsigned long long* host8, int reset) {
    if (host8 && cudaMemcpyFromSymbol(host8, g_nn_wait, sizeof(unsigned long long) * 8) != cudaSuccess) return PDP_ERR_CUDA;
    (void)0;
    if (reset) { unsigned long long z[8] = {0}; if (cudaMemcpyToSymbol(g_nn_wait, z, sizeof(z)) != cudaSuccess) return PDP_ERR_CUDA; }
    return PDP_OK;
}
#endif

// K elements per chunk of the weight image (the host side builds the images accordingly)
extern "C" int pdp_edge_nn_chunk_k(void) { return kChunkK; }
// 1: the weight images are rows of 64 bytes with the 16-byte units of row n at unit ^ ((n >> 1) & 3); 0: column groups of [n_tot][16 bytes]
extern "C" int pdp_edge_nn_swizzle(void) { return 1; }
static_assert(kChunkK == 16, "the operand staging and the 64-byte swizzle are written for 16-element K chunks");

extern "C" int pdp_edge_mlp_forward(const float* x1, int32_t k1, const float* x2, int32_t k2, const float* x3, int32_t k3, int64_t rows,
                                    const float* w_img, const float* bias, int32_t n_blk, int32_t n_mma, int32_t passes, int32_t n_out,
                                    int32_t act, const float* row_mask, float* out, void* stream) {
    if (rows <= 0) return PDP_OK;
    EdgeNNArgs P;
    memset(&P, 0, sizeof(P));
    if (!fill_common(P, x1, k1, x2, k2, x3, k3, rows, w_img, bias, n_blk, n_mma, passes, "pdp_edge_mlp_forward")) return PDP_ERR_ARG;
    if (!out || n_out < 1 || n_out > passes * P.n_tot || P.n_tot > 256) { pdp_set_error("pdp_edge_mlp_forward: bad output shape"); return PDP_ERR_ARG; }
    P.n_out = n_out; P.act = act; P.row_mask = row_mask; P.out = out;
    {
        const size_t stage = 2u * kTileM * kChunkK * 4u + 2u * (size_t)P.n_tot * kChunkK * 4u;
        const char* e = getenv("PDP_B200_NN_OTILE");      // (profiling: 0 = thread-per-row stores)
        P.out_tile = passes == 1 && !((uintptr_t)out & 15) && stage * P.stages + kRawBytes + (size_t)kTileM * n_out * 4 <= 227 * 1024 &&
                     !(e && atoi(e) == 0);
    }
    return launch(P, EPI_LINEAR, (cudaStream_t)stream);
}

// torch.nn.GRUCell over rows: h'[rows, H] from input [x1 | x2] and hidden state h (row-major [rows, H]); every pass holds
// n_blk * n_mma / 4 hidden units, four accumulator columns each (r, z, W_in x, W_hn h).  row_mask blends h' with h (frozen rows).
extern "C" int pdp_edge_gru_forward(const float* x1, int32_t k1, const float* x2, int32_t k2, const float* h, int32_t hidden, int64_t rows,
                                    const float* w_img, const float* bias, int32_t n_blk, int32_t n_mma, int32_t passes,
                                    const float* row_mask, float* out, void* stream) {
    if (rows <= 0) return PDP_OK;
    EdgeNNArgs P;
    memset(&P, 0, sizeof(P));
    if (!fill_common(P, h, hidden, x1, k1, x2, k2, rows, w_img, bias, n_blk, n_mma, passes, "pdp_edge_gru_forward")) return PDP_ERR_ARG;   // rows = [h | x1 | x2]
    if (!out || !h || hidden < 1 || (P.n_tot & 15) || hidden > passes * (P.n_tot / 4) || out == h) {
        pdp_set_error("pdp_edge_gru_forward: bad shape (hidden=%d n_tot=%d passes=%d) or out aliases h", hidden, P.n_tot, passes);
        return PDP_ERR_ARG;
    }
    P.n_out = hidden; P.row_mask = row_mask; P.h_old = h; P.out = out;
    return launch(P, EPI_GRU, (cudaStream_t)stream);
}
