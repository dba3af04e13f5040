// Phi(Phi^T V): the kernel matvec GPyTorch's conjugate gradients call (K3 + K5 + K6
// in SURVEY.md 2a), with the modulator f_l applied at matvec time.
//
// Replaces, per matvec, in the reference:
//   2L x SparseLinearOperator._matmul          utils_sparse/sparse_lo.py:16-18  (cuSPARSE SpMM, int64 indices)
//   L  x .t().to_sparse_csr()                  utils_sparse/sparse_lo.py:23-25
//   2L scalar*matrix + 2(L-1) adds on N x t    gptorch_kernels_sparse/sparse_grf_kernel.py:59-61
//   scatter / gather of the selected rows      gptorch_kernels_sparse/sparse_grf_kernel.py:32-41
//
// Both halves are the same operation on block-CSR data ("for every row, for
// every walk length l, f_l * sum of val * X[col, :]"), once over Phi^T blocks
// (U = Phi[x2]^T V) and once over Phi blocks (out = Phi[x1] U):
//   * entries are 8-byte {length<<27 | col, val} pairs streamed once, coalesced;
//   * TPR threads share a row and own 4 (or 1) of the t right-hand-side
//     columns each, so a gather of X[col, :] is one 16*TPR-byte contiguous read;
//   * f_l is applied per entry in registers (f lives in shared memory).
// HBM-bound: algorithmic bytes per matvec = 2*nnz*8 + 2*L*(rows+1)*4 + 4*N*t*4
// (SURVEY.md 8d); the X gathers are L2/L1 traffic.  No tensor cores: this is a
// sparse gather, not a dense contraction.

#include "grf_common.cuh"

// Tuned on config 2 (t = 16, merged Phi_f; CUDA events, L2 flushed): (min CTAs/SM, gathers in flight per lane)
//   (5,4) 74.5 us   (4,8) 62.5   (4,4) 56.0   (3,4) 55.8   (3,8) 56.1   (2,16) 51.9  <- fewer, fatter warps win
#ifndef GRF_SPMM_MINBLOCKS
#define GRF_SPMM_MINBLOCKS 2  // resident CTAs of 256 threads per SM the register budget allows (<= 128 registers)
#endif
#ifndef GRF_SPMM_BATCH
#define GRF_SPMM_BATCH 16     // independent gathers in flight per lane
#endif
#ifndef GRF_SPMM_STATIC_PCT
#define GRF_SPMM_STATIC_PCT 50  // share of a pass's row groups assigned by fixed stride; the rest goes by ticket
// (R-MAT 2^20 nodes, per-length matvec: fixed stride 2.92 ms, 90 % 2.73, 75 % 2.60, 50 % 2.48, 0 % 2.49; config 2: 52.3 us for all)
#endif

namespace grf {

// one or two lanes per row (t <= 8) keep little state per row: there more resident warps win
// (t = 1: 33.8 us at 3 CTAs/SM and 8 gathers in flight against 66 us at 2 CTAs/SM)
__host__ __device__ constexpr int spmm_min_blocks(int tpr) { return tpr >= 4 ? GRF_SPMM_MINBLOCKS : 3; }
__host__ __device__ constexpr int spmm_batch(int tpr) { return tpr >= 4 ? GRF_SPMM_BATCH : 8; }

template <int VEC>
struct Vec;
template <>
struct Vec<4> {
    float4 v;
    __device__ __forceinline__ void zero() { v = make_float4(0.f, 0.f, 0.f, 0.f); }
    __device__ __forceinline__ void load(const float *p) { v = __ldg(reinterpret_cast<const float4 *>(p)); }
    // gathered once, never again from this SM: do not allocate the line in L1 (a miss then costs one pass
    // through the L1 data stage instead of two -- fill, then read; ncu on the power-law Phi: 1.75
    // wavefronts per gathered entry at a 27 % hit rate)
    __device__ __forceinline__ void load_stream(const float *p) {
        // (ld.global.cg instead: Phi^T V 12.9 ms, Phi U 25.6 ms against 5.4 / 5.0 ms with cached loads at config 4)
        asm volatile("ld.global.nc.L1::no_allocate.v4.f32 {%0, %1, %2, %3}, [%4];"
                     : "=f"(v.x), "=f"(v.y), "=f"(v.z), "=f"(v.w)
                     : "l"(p));
    }
    __device__ __forceinline__ void load_shared(const float *p) { v = *reinterpret_cast<const float4 *>(p); }
    __device__ __forceinline__ void store(float *p) const { *reinterpret_cast<float4 *>(p) = v; }
    __device__ __forceinline__ void add_from(const float *p, int ncols, bool vec_ok) {
        if (ncols >= 4 && vec_ok) {
            const float4 o = *reinterpret_cast<const float4 *>(p);
            v.x += o.x; v.y += o.y; v.z += o.z; v.w += o.w;
        } else {
            v.x += p[0];
            if (ncols > 1) v.y += p[1];
            if (ncols > 2) v.z += p[2];
            if (ncols > 3) v.w += p[3];
        }
    }
    // first `ncols` (1..4) columns; vector store only when all four are valid and p is 16-byte aligned
    __device__ __forceinline__ void store_cols(float *p, int ncols, bool vec_ok) const {
        if (ncols >= 4 && vec_ok) {
            store(p);
        } else {
            p[0] = v.x;
            if (ncols > 1) p[1] = v.y;
            if (ncols > 2) p[2] = v.z;
            if (ncols > 3) p[3] = v.w;
        }
    }
    __device__ __forceinline__ void fma(float a, const Vec &x) {
        v.x = fmaf(a, x.v.x, v.x);
        v.y = fmaf(a, x.v.y, v.y);
        v.z = fmaf(a, x.v.z, v.z);
        v.w = fmaf(a, x.v.w, v.w);
    }
    __device__ __forceinline__ float dot(const Vec &x) const {
        return v.x * x.v.x + v.y * x.v.y + v.z * x.v.z + v.w * x.v.w;
    }
};
template <>
struct Vec<1> {
    float v;
    __device__ __forceinline__ void zero() { v = 0.f; }
    __device__ __forceinline__ void load(const float *p) { v = __ldg(p); }
    __device__ __forceinline__ void load_stream(const float *p) {
        asm volatile("ld.global.nc.L1::no_allocate.f32 %0, [%1];" : "=f"(v) : "l"(p));
    }
    __device__ __forceinline__ void load_shared(const float *p) { v = *p; }
    __device__ __forceinline__ void store(float *p) const { *p = v; }
    __device__ __forceinline__ void add_from(const float *p, int, bool) { v += *p; }
    __device__ __forceinline__ void store_cols(float *p, int, bool) const { *p = v; }
    __device__ __forceinline__ void fma(float a, const Vec &x) { v = fmaf(a, x.v, v); }
    __device__ __forceinline__ float dot(const Vec &x) const { return v * x.v; }
};

__device__ __forceinline__ GrfEntry load_entry(const GrfEntry *p) {
    const int2 raw = __ldg(reinterpret_cast<const int2 *>(p));
    GrfEntry e;
    e.col = raw.x;
    e.val = __int_as_float(raw.y);
    return e;
}

// Y[k, :] = sum_{e in row_k} f[step(e)] * e.val * X[col(e), :]
//
// A row's L per-length segments are contiguous, so the whole row is ONE flat
// run of entries [ptr[row*L], ptr[(row+1)*L]) with the length packed in the
// top bits of `col`.  TPR lanes own a row.  Per round the group fetches
// TPR*kEPL entries with one coalesced 8-byte load per lane and entry slot
// (all independent), scales them by f[length] in registers, and then every
// lane replays the group's entries through width-TPR shuffles, issuing the
// X[col, :] gathers back to back (TPR*kEPL independent 16-byte loads per lane
// in flight).  The next round's entries are prefetched before the gathers of
// the current one are consumed, so entry-stream latency hides behind the
// gather latency.  (v1 walked entry -> gather serially: ncu showed 25 warps
// stalled on long-scoreboard per issue and 0.42 entries/cycle/SM.)
// entries per lane per round: a round covers TPR * epl(TPR) entry slots -- 16 for 4..16 lanes per
// row (rows of the merged Phi average ~28 entries at config 2; more slots only add padding)
__host__ __device__ constexpr int epl(int tpr) { return tpr >= 16 ? 1 : (tpr >= 4 ? 16 / tpr : 4); }

// One row for the TPR lanes that own it.  `X` is either global memory (ldx = leading
// dimension) or, for the tiled kernel, the shared-memory copy of X[cmin .. cmax, :]
// (then `col_off` = cmin).  Returns the accumulator of this lane's VEC columns.
//
// All 32 lanes of the warp call this together and run the same number of rounds (the
// longest row of the warp's 32/TPR rows decides), so every shuffle uses the constant full
// mask: with a per-group mask nvcc expands each __shfl_sync into a MATCH/REDUX/VOTE loop
// (ncu: ~10 extra instructions per shuffle, 4.6 warp-instructions per entry).
constexpr int kGatherCached = 0, kGatherShared = 1, kGatherStream = 2;
template <int TPR, int VEC, int kMode>
__device__ __forceinline__ Vec<VEC> spmm_row(const int2 *__restrict__ ent2, int32_t b, int32_t e,
                                             int2 (&nxt)[epl(TPR)], int32_t next_b, int32_t next_e,
                                             const float *__restrict__ fs, const float *X, uint32_t ldx,
                                             int32_t col_off, int c0, bool live, int sub) {
    // X offsets are 32-bit element counts, multiplied by the leading dimension once per entry when it is
    // staged (not once per lane and gather): the 64-bit col * ldx + c0 arithmetic was 8 of the ~20
    // instructions per gathered entry (ncu instruction mix: IMAD 19 %, LEA 10 %, SHF 6 %).  The host
    // falls back to the plain kernel when rows(X) * ldx does not fit in 32 bits.
    // `nxt` holds the row's first round of entries on entry; on exit it holds the first round
    // of the NEXT row of this group ([next_b, next_e)), fetched while the last gathers of this
    // row are in flight -- a two-deep software pipeline across rows (ncu on the one-row-at-a-
    // time version: 10 warps stalled on long scoreboard per issue, L1 pipe only 40 % busy).
    constexpr unsigned gmask = 0xffffffffu;
    constexpr int kEPL = epl(TPR);
    const int32_t b_end = b + __reduce_max_sync(0xffffffffu, e - b);  // warp-uniform trip count
    Vec<VEC> acc;
    acc.zero();
    int32_t base = b;
    do {
        uint32_t cl[kEPL];
        float sv[kEPL];
#pragma unroll
        for (int q = 0; q < kEPL; ++q) {
            // a padding slot is the all-zero pair: gather row col_off (always valid) with weight 0
            const bool pad = (nxt[q].x | nxt[q].y) == 0;
            cl[q] = pad ? 0u : (((uint32_t)nxt[q].x & kColMask) - (uint32_t)col_off) * ldx;
            sv[q] = __int_as_float(nxt[q].y) * fs[(uint32_t)nxt[q].x >> kStepShift];
        }
        const int32_t nb = base + TPR * kEPL;
        if (nb < b_end) {
#pragma unroll
            for (int q = 0; q < kEPL; ++q) {
                const int32_t idx = nb + q * TPR + sub;
                nxt[q] = idx < e ? __ldg(ent2 + idx) : make_int2(0, 0);
            }
        } else {
#pragma unroll
            for (int q = 0; q < kEPL; ++q) {
                const int32_t idx = next_b + q * TPR + sub;
                nxt[q] = idx < next_e ? __ldg(ent2 + idx) : make_int2(0, 0);
            }
        }
        // Gathers in batches of kBatch independent loads, all unconditional and in bounds
        // (padding slots read row `col_off` with weight 0): with the loads predicated per
        // entry nvcc re-used one register quad and serialised load -> FMA -> load (ncu: one
        // long-scoreboard stall per entry, 16 dependent L2 round trips per round).
        constexpr int kSlots = TPR * kEPL;
        constexpr int kBatch = kSlots < spmm_batch(TPR) ? kSlots : spmm_batch(TPR);
#pragma unroll
        for (int m0 = 0; m0 < kSlots; m0 += kBatch) {
            Vec<VEC> x[kBatch];
            float a[kBatch];
#pragma unroll
            for (int m = 0; m < kBatch; ++m) {
                const int q = (m0 + m) / TPR, j = (m0 + m) % TPR;
                const uint32_t off = TPR == 1 ? cl[q] : __shfl_sync(gmask, cl[q], j, TPR);
                a[m] = TPR == 1 ? sv[q] : __shfl_sync(gmask, sv[q], j, TPR);
                if (kMode == kGatherShared)
                    x[m].load_shared(X + (off + (uint32_t)c0));
                else if (kMode == kGatherStream)
                    x[m].load_stream(X + (off + (uint32_t)c0));
                else
                    x[m].load(X + (off + (uint32_t)c0));
            }
#pragma unroll
            for (int m = 0; m < kBatch; ++m) acc.fma(a[m], x[m]);
        }
        base = nb;
    } while (base < b_end);
    return acc;
}

template <int TPR>
__device__ __forceinline__ void load_first_round(const int2 *__restrict__ ent2, int32_t b, int32_t e, int sub,
                                                 int2 (&nxt)[epl(TPR)]) {
    constexpr int kEPL = epl(TPR);
#pragma unroll
    for (int q = 0; q < kEPL; ++q) {
        const int32_t idx = b + q * TPR + sub;
        nxt[q] = idx < e ? __ldg(ent2 + idx) : make_int2(0, 0);
    }
}

template <int TPR, int VEC, bool kStream = false>
__global__ void __launch_bounds__(256, spmm_min_blocks(TPR)) spmm_blocks_kernel(const int32_t *__restrict__ ptr,
                                                          const GrfEntry *__restrict__ ent,
                                                          const float *__restrict__ f, int32_t L,
                                                          const int32_t *__restrict__ row_ids, int64_t n_tasks,
                                                          int64_t row_lo, int64_t n_rows,
                                                          const float *__restrict__ X, int64_t ldx,
                                                          float *__restrict__ Y, int64_t ldy, int32_t t,
                                                          int32_t t_store, int32_t vec_store, int32_t long_thresh,
                                                          const int2 *__restrict__ chunk_bounds,
                                                          int32_t out_by_row, int32_t *__restrict__ sched,
                                                          int32_t accumulate) {
    // sched != NULL: {ticket, finished warps}, both zero at launch and zero again at exit.  The first
    // GRF_SPMM_STATIC_PCT % of the row groups go to the warps by fixed stride (neighbouring rows stay
    // on one SM), the rest by an atomic ticket fetched one iteration ahead: with skewed row lengths
    // (power-law graphs) a fixed stride leaves SMs idle at the end (R-MAT 2^20: 2.92 -> 2.48 ms per
    // product); on the uniform rows of config 2 it changes nothing.
    // out_by_row: row_ids lists the non-empty rows and task k writes Y[row_ids[k]] (Phi^T of a row
    // shard touches only a fraction of the N columns); otherwise task k writes Y[k].
    // t = columns computed (a multiple of VEC; the operands are padded to it), t_store <= t = columns
    // that exist in Y; vec_store: rows of Y are 16-byte aligned (16-byte stores allowed).
    // long_thresh > 0: rows with more entries are left to the chunk launch (hub columns of a
    // power-law Phi^T hold 10^5..10^6 entries; one 4-lane group would serialise them);
    // chunk_bounds != NULL: this IS the chunk launch -- task k is the entry range chunk_bounds[k]
    // and its partial sum goes to row k of Y (the caller's partial buffer).
    __shared__ float fs[kMaxSteps];
    if (threadIdx.x < kMaxSteps) fs[threadIdx.x] = threadIdx.x < L ? __ldg(f + threadIdx.x) : 0.f;
    __syncthreads();
    const int sub = threadIdx.x % TPR;
    constexpr int kGroupsPerWarp = 32 / TPR;
    const int g_in_warp = (threadIdx.x & 31) / TPR;
    const int64_t warp0 = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    const int64_t warp_stride = ((int64_t)gridDim.x * blockDim.x) >> 5;
    const int2 *ent2 = reinterpret_cast<const int2 *>(ent);
    const int n_tiles = (t + TPR * VEC - 1) / (TPR * VEC);
    // warp-uniform loop: the warp takes 32/TPR consecutive tasks per iteration; the row bounds of
    // the next iteration are fetched one iteration ahead, its first entries by spmm_row
    auto bounds = [&](int64_t k, int32_t &b, int32_t &e, bool &mine, int64_t &orow) {
        b = e = 0;
        orow = k;
        if (chunk_bounds) {
            // chunk launch: row_ids, when given, is the order in which the chunks are issued (GrfLongRows.chunk_order)
            mine = k < n_tasks;
            if (mine) {
                const int64_t c = row_ids ? (int64_t)__ldg(row_ids + k) : k;
                const int2 be = __ldg(chunk_bounds + c);
                b = be.x;
                e = be.y;
                orow = c;
            }
            return;
        }
        int64_t row = -1;
        if (k < n_tasks) row = row_ids ? (int64_t)__ldg(row_ids + k) - row_lo : k;
        mine = row >= 0 && row < n_rows;  // ids outside this shard are skipped
        if (out_by_row) orow = row;
        if (mine) {
            b = __ldg(ptr + row * L);
            e = __ldg(ptr + (row + 1) * L);
            if (long_thresh > 0 && e - b > long_thresh) {
                mine = false;  // split row: written by long_reduce_kernel
                e = b;
            }
        }
    };
    // iteration `it` = the 32/TPR consecutive tasks [it * G, (it + 1) * G) of one warp
    const int lane = threadIdx.x & 31;
    const int32_t n_warps = (int32_t)warp_stride;
    const int32_t n_iters = (int32_t)((n_tasks + kGroupsPerWarp - 1) / kGroupsPerWarp);
    // Iterations [0, n_static) are assigned up front, the rest by ticket.  The static part gives
    // every SM ONE contiguous range of rows, which its resident warps walk interleaved (warp j of
    // the SM takes range_begin + j, + warps_per_sm, ...): at any moment an SM works on ~128
    // consecutive rows and its window of X slides, so a banded Phi re-reads X from L1, not L2
    // (with a grid-wide stride every iteration of a warp landed in a fresh window).
    const int32_t n_static = sched ? (int32_t)((int64_t)n_iters * GRF_SPMM_STATIC_PCT / 100) : n_iters;
    int32_t it, it_step, it_end;
    // (an ordered chunk launch wants the opposite: all SMs advance through the order together, so that the
    // chunks in flight share one window of X in L2 -> plain grid stride)
    if (gridDim.x % kSmCount == 0 && !(chunk_bounds && row_ids)) {
        const int warps_per_block = blockDim.x >> 5;
        const int per_sm = gridDim.x / kSmCount;
        // CTAs are handed to the SMs round-robin, so blockIdx = s, s + 148, ... share an SM and its L1
        // (only a locality hint: correctness does not depend on the placement)
        const int sm = blockIdx.x % kSmCount;
        const int32_t q = (n_static + kSmCount - 1) / kSmCount;
        it = sm * q + (blockIdx.x / kSmCount) * warps_per_block + (threadIdx.x >> 5);
        it_step = per_sm * warps_per_block;
        it_end = min((sm + 1) * q, n_static);
    } else {
        it = (int32_t)warp0;
        it_step = n_warps;
        it_end = n_static;
    }
    auto finish = [&]() {
        if (sched && lane == 0) {
            if (atomicAdd(sched + 1, 1) == n_warps - 1) {  // every other warp has drawn its last ticket
                sched[0] = 0;
                sched[1] = 0;
            }
        }
    };
    auto ticket = [&]() {
        int32_t tk = 0;
        if (lane == 0) tk = n_static + atomicAdd(sched, 1);
        return __shfl_sync(0xffffffffu, tk, 0);
    };
    bool static_next = true;  // `itn` still belongs to this warp's static sequence
    if (it >= it_end) {
        it = sched ? ticket() : n_iters;
        static_next = false;
    }
    if (it >= n_iters) {
        finish();
        return;
    }
    int32_t itn;
    if (static_next && it + it_step < it_end) {
        itn = it + it_step;
    } else {
        itn = sched ? ticket() : n_iters;
        static_next = false;
    }
    int32_t b, e, nb, ne;
    bool mine, nmine;
    int64_t orow, norow;
    bounds((int64_t)it * kGroupsPerWarp + g_in_warp, b, e, mine, orow);
    int2 nxt[epl(TPR)];
    load_first_round<TPR>(ent2, b, e, sub, nxt);
    while (it < n_iters) {
        // the iteration after next: the next one of the static sequence, or a ticket whose latency
        // this iteration hides
        const int32_t after = static_next && itn + it_step < it_end ? itn + it_step : -1;
        const bool draw = sched && after < 0;
        int32_t tk = 0;
        if (draw && lane == 0) tk = n_static + atomicAdd(sched, 1);
        bounds((int64_t)itn * kGroupsPerWarp + g_in_warp, nb, ne, nmine, norow);
        for (int tile = 0; tile < n_tiles; ++tile) {
            // lanes whose columns fall outside t (t not a multiple of TPR*VEC) still help with the
            // entry loads and shuffles; they just do not gather or store
            const int c0 = (tile * TPR + sub) * VEC;
            const bool live = mine && c0 < t;
            const bool last_tile = tile + 1 == n_tiles;
            Vec<VEC> acc = spmm_row<TPR, VEC, kStream ? kGatherStream : kGatherCached>(
                ent2, b, e, nxt, last_tile ? nb : b, last_tile ? ne : e, fs, X, (uint32_t)ldx, 0, c0 < t ? c0 : 0, live,
                sub);
            if (live && c0 < t_store) {
                // accumulate: Y += (the second and later row blocks of a block-wise Phi^T add to U)
                if (accumulate) acc.add_from(Y + orow * ldy + c0, t_store - c0, vec_store != 0);
                acc.store_cols(Y + orow * ldy + c0, t_store - c0, vec_store != 0);
            }
        }
        b = nb;
        e = ne;
        mine = nmine;
        orow = norow;
        it = itn;
        if (after >= 0) {
            itn = after;
        } else {
            itn = draw ? __shfl_sync(0xffffffffu, tk, 0) : n_iters;
            static_next = false;
        }
    }
    finish();
}

// Tiled variant for banded Phi (lattices, rings, any ordering with locality): a CTA owns
// `chunk_rows` consecutive rows; the union of their column windows (precomputed per 32
// rows by grf_block_windows) is copied once, coalesced, into shared memory -- up to
// 224 KB of X -- and every gather of the chunk is then a shared-memory read: half the
// L1 wavefronts per entry of a global gather, no tag lookups, no L2 round trips.  A
// chunk whose window does not fit (long-range edges) takes the global-gather path.
template <int TPR>
__global__ void __launch_bounds__(512, 1) spmm_tiled_kernel(const int32_t *__restrict__ ptr,
                                                             const GrfEntry *__restrict__ ent,
                                                             const float *__restrict__ f, int32_t L,
                                                             int64_t n_rows, int32_t chunk_rows,
                                                             const int2 *__restrict__ win, int32_t cap_rows,
                                                             const float *__restrict__ X, int64_t ldx,
                                                             float *__restrict__ Y, int64_t ldy, int32_t t) {
    extern __shared__ __align__(16) float tile[];
    __shared__ float fs[kMaxSteps];
    __shared__ int s_min, s_max;
    if (threadIdx.x < kMaxSteps) fs[threadIdx.x] = threadIdx.x < L ? __ldg(f + threadIdx.x) : 0.f;
    const int sub = threadIdx.x % TPR;
    const int gid = threadIdx.x / TPR;
    const int ngroups = blockDim.x / TPR;
    const int g_in_warp = (threadIdx.x & 31) / TPR;
    const int2 *ent2 = reinterpret_cast<const int2 *>(ent);
    const int c0 = sub * 4 < t ? sub * 4 : 0;  // lanes beyond t read column 0 and do not store
    const bool col_live = sub * 4 < t;
    const int ldt = (t + 3) & ~3;  // tile leading dimension (floats)
    const int64_t n_chunks = (n_rows + chunk_rows - 1) / chunk_rows;
    for (int64_t chunk = blockIdx.x; chunk < n_chunks; chunk += gridDim.x) {
        const int64_t r0 = chunk * chunk_rows;
        const int64_t r1 = min(n_rows, r0 + chunk_rows);
        if (threadIdx.x == 0) {
            s_min = 0x7fffffff;
            s_max = -1;
        }
        __syncthreads();
        for (int64_t g = r0 / 32 + threadIdx.x; g <= (r1 - 1) / 32; g += blockDim.x) {
            const int2 w = __ldg(win + g);
            if (w.y >= w.x) {
                atomicMin(&s_min, w.x);
                atomicMax(&s_max, w.y);
            }
        }
        __syncthreads();
        const int cmin = s_min, cmax = s_max;
        const int width = cmax - cmin + 1;
        const bool tiled = width > 0 && width <= cap_rows;
        if (tiled) {
            const int vec_per_row = ldt >> 2;
            const int n_vec = width * vec_per_row;
            for (int i = threadIdx.x; i < n_vec; i += blockDim.x) {
                const int r = i / vec_per_row, q = i - r * vec_per_row;
                const float4 v = __ldg(reinterpret_cast<const float4 *>(X + (int64_t)(cmin + r) * ldx) + q);
                reinterpret_cast<float4 *>(tile)[i] = v;
            }
        }
        __syncthreads();
        // warp-uniform loop over the chunk's rows (32/TPR consecutive rows per warp and iteration)
        auto bounds = [&](int64_t row, int32_t &b, int32_t &e) {
            b = e = 0;
            if (row < r1) {
                b = __ldg(ptr + row * L);
                e = __ldg(ptr + (row + 1) * L);
            }
        };
        int64_t rb = r0 + gid - g_in_warp;
        if (rb < r1) {
            int32_t b, e, nb, ne;
            bounds(rb + g_in_warp, b, e);
            int2 nxt[epl(TPR)];
            load_first_round<TPR>(ent2, b, e, sub, nxt);
            for (; rb < r1; rb += ngroups) {
                const int64_t row = rb + g_in_warp;
                bounds(row + ngroups, nb, ne);
                const bool live = row < r1 && col_live;
                Vec<4> acc;
                if (tiled)
                    acc = spmm_row<TPR, 4, kGatherShared>(ent2, b, e, nxt, nb, ne, fs, tile, (uint32_t)ldt, cmin, c0, live, sub);
                else
                    acc = spmm_row<TPR, 4, kGatherCached>(ent2, b, e, nxt, nb, ne, fs, X, (uint32_t)ldx, 0, c0, live, sub);
                if (live) acc.store(Y + row * ldy + c0);
                b = nb;
                e = ne;
            }
        }
        __syncthreads();
    }
}

// Column window [min col, max col] of every group of 32 consecutive rows (one warp each),
// and the widest window over all groups (atomicMax into *max_width).
__global__ void __launch_bounds__(256) block_windows_kernel(const int32_t *__restrict__ ptr,
                                                            const GrfEntry *__restrict__ ent, int64_t n_rows,
                                                            int32_t L, int2 *__restrict__ win,
                                                            int32_t *__restrict__ max_width) {
    const int lane = threadIdx.x & 31;
    const int64_t warp0 = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    const int64_t nwarps = ((int64_t)gridDim.x * blockDim.x) >> 5;
    const int64_t n_groups = (n_rows + 31) / 32;
    for (int64_t g = warp0; g < n_groups; g += nwarps) {
        const int64_t r0 = g * 32, r1 = min(n_rows, r0 + 32);
        const int32_t b = __ldg(ptr + r0 * L), e = __ldg(ptr + r1 * L);
        int lo = 0x7fffffff, hi = -1;
        for (int32_t i = b + lane; i < e; i += 32) {
            const int c = (int)((uint32_t)ent[i].col & kColMask);
            lo = min(lo, c);
            hi = max(hi, c);
        }
#pragma unroll
        for (int d = 16; d > 0; d >>= 1) {
            lo = min(lo, __shfl_xor_sync(0xffffffffu, lo, d));
            hi = max(hi, __shfl_xor_sync(0xffffffffu, hi, d));
        }
        if (lane == 0) {
            win[g] = make_int2(lo, hi);
            if (hi >= lo) atomicMax(max_width, hi - lo + 1);
        }
    }
}

// Few right-hand sides (t <= 4: Thompson sampling draws one posterior sample, bo_utils.py:272): G lanes
// share a row and take DIFFERENT entries (CSR-vector), each gathering all t columns of X[col, :], and
// reduce with shuffles at the end.  Entry loads are coalesced across the group and a long row (a BO
// training row holds up to 1 + (L-1) W entries) is spread over 8 or 32 lanes instead of one.
template <int G, int T>
__global__ void __launch_bounds__(256) spmv_coop_kernel(const int32_t *__restrict__ ptr,
                                                        const GrfEntry *__restrict__ ent,
                                                        const float *__restrict__ f, int32_t L,
                                                        const int32_t *__restrict__ row_ids, int64_t n_tasks,
                                                        int64_t row_lo, int64_t n_rows, const float *__restrict__ X,
                                                        int64_t ldx, float *__restrict__ Y, int64_t ldy,
                                                        int32_t long_thresh, const int2 *__restrict__ chunk_bounds,
                                                        int32_t out_by_row, int32_t accumulate) {
    __shared__ float fs[kMaxSteps];
    if (threadIdx.x < kMaxSteps) fs[threadIdx.x] = threadIdx.x < L ? __ldg(f + threadIdx.x) : 0.f;
    __syncthreads();
    const int sub = threadIdx.x % G;
    constexpr int kGroupsPerWarp = 32 / G;
    const int g_in_warp = (threadIdx.x & 31) / G;
    const int64_t warp0 = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    const int64_t warp_stride = ((int64_t)gridDim.x * blockDim.x) >> 5;
    const int2 *ent2 = reinterpret_cast<const int2 *>(ent);
    for (int64_t kb = warp0 * kGroupsPerWarp; kb < n_tasks; kb += warp_stride * kGroupsPerWarp) {
        const int64_t k = kb + g_in_warp;
        int32_t b = 0, e = 0;
        bool mine = false;
        int64_t orow = k;
        if (chunk_bounds) {
            mine = k < n_tasks;
            if (mine) {
                const int2 be = __ldg(chunk_bounds + k);
                b = be.x;
                e = be.y;
            }
        } else {
            int64_t row = -1;
            if (k < n_tasks) row = row_ids ? (int64_t)__ldg(row_ids + k) - row_lo : k;
            mine = row >= 0 && row < n_rows;
            if (out_by_row) orow = row;
            if (mine) {
                b = __ldg(ptr + row * L);
                e = __ldg(ptr + (row + 1) * L);
                if (long_thresh > 0 && e - b > long_thresh) {
                    mine = false;
                    e = b;
                }
            }
        }
        float acc[T];
#pragma unroll
        for (int j = 0; j < T; ++j) acc[j] = 0.f;
        constexpr int kU = 4;  // entries in flight per lane
        for (int32_t i0 = b + sub; i0 < e; i0 += G * kU) {
            int2 raw[kU];
#pragma unroll
            for (int u = 0; u < kU; ++u) {
                const int32_t i = i0 + u * G;
                raw[u] = i < e ? __ldg(ent2 + i) : make_int2(0, 0);
            }
            float x[kU][T];
#pragma unroll
            for (int u = 0; u < kU; ++u) {
                const float *src = X + (int64_t)((uint32_t)raw[u].x & kColMask) * ldx;  // padding reads row 0
#pragma unroll
                for (int j = 0; j < T; ++j) x[u][j] = __ldg(src + j);
            }
#pragma unroll
            for (int u = 0; u < kU; ++u) {
                const float a = __int_as_float(raw[u].y) * fs[(uint32_t)raw[u].x >> kStepShift];
#pragma unroll
                for (int j = 0; j < T; ++j) acc[j] = fmaf(a, x[u][j], acc[j]);
            }
        }
#pragma unroll
        for (int d = G / 2; d > 0; d >>= 1) {
#pragma unroll
            for (int j = 0; j < T; ++j) acc[j] += __shfl_xor_sync(0xffffffffu, acc[j], d);
        }
        if (mine && sub == 0) {
#pragma unroll
            for (int j = 0; j < T; ++j) Y[orow * ldy + j] = accumulate ? Y[orow * ldy + j] + acc[j] : acc[j];
        }
    }
}

// vfull[(x2[k] - row_lo), :] += v[k, :]   (vfull zeroed by the caller)
__global__ void __launch_bounds__(256) scatter_rows_kernel(const int32_t *__restrict__ x2, int64_t n2,
                                                           int64_t row_lo, int64_t n_rows,
                                                           const float *__restrict__ v, int64_t ldv,
                                                           float *__restrict__ vfull, int64_t ldu, int32_t t) {
    const int64_t total = n2 * t;
    for (int64_t g = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; g < total;
         g += (int64_t)gridDim.x * blockDim.x) {
        const int64_t k = g / t;
        const int c = (int)(g - k * t);
        const int64_t row = (int64_t)__ldg(x2 + k) - row_lo;
        if (row < 0 || row >= n_rows) continue;
        atomicAdd(vfull + row * ldu + c, __ldg(v + k * ldv + c));
    }
}

// vfull[r, 0:t] = v[r, 0:t] for all rows (staging a V whose rows are not 16-byte friendly; a 2-D
// DMA copy with 4*t-byte rows is far slower than this)
__global__ void __launch_bounds__(256) pad_copy_kernel(const float *__restrict__ v, int64_t ldv,
                                                       float *__restrict__ vfull, int64_t ldu, int64_t n_rows,
                                                       int32_t t) {
    const int64_t total = n_rows * t;
    for (int64_t g = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; g < total;
         g += (int64_t)gridDim.x * blockDim.x) {
        const int64_t r = g / t;
        const int c = (int)(g - r * t);
        vfull[r * ldu + c] = __ldg(v + r * ldv + c);
    }
}

// same without atomics, for index sets without repeated ids (rows outside x2 keep their zeros)
__global__ void __launch_bounds__(256) scatter_rows_unique_kernel(const int32_t *__restrict__ x2, int64_t n2,
                                                                  int64_t row_lo, int64_t n_rows,
                                                                  const float *__restrict__ v, int64_t ldv,
                                                                  float *__restrict__ vfull, int64_t ldu,
                                                                  int32_t t) {
    const int64_t total = n2 * t;
    for (int64_t g = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; g < total;
         g += (int64_t)gridDim.x * blockDim.x) {
        const int64_t k = g / t;
        const int c = (int)(g - k * t);
        const int64_t row = (int64_t)__ldg(x2 + k) - row_lo;
        if (row < 0 || row >= n_rows) continue;
        vfull[row * ldu + c] = __ldg(v + k * ldv + c);
    }
}

// U[col, :] += f[l] * val * V[k, :] for every entry of row x2[k] -- the first half of the product
// when x2 is a small subset of the rows (a BO training set of 10^2..10^3 nodes out of 10^5..10^6):
// work proportional to the selected rows instead of one pass over all of Phi^T.  fp32 atomics:
// the summation order, hence the last bits, can differ between runs.
__global__ void __launch_bounds__(256) spmm_scatter_kernel(const int32_t *__restrict__ ptr,
                                                           const GrfEntry *__restrict__ ent,
                                                           const float *__restrict__ f, int32_t L,
                                                           const int32_t *__restrict__ x2, int64_t n2,
                                                           int64_t row_lo, int64_t n_rows,
                                                           const float *__restrict__ V, int64_t ldv,
                                                           float *__restrict__ U, int64_t ldu, int32_t t) {
    // one warp per selected row; lanes take different entries (coalesced), each adds all t columns
    __shared__ float fs[kMaxSteps];
    if (threadIdx.x < kMaxSteps) fs[threadIdx.x] = threadIdx.x < L ? __ldg(f + threadIdx.x) : 0.f;
    __syncthreads();
    const int lane = threadIdx.x & 31;
    const int64_t warp0 = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    const int64_t nwarps = ((int64_t)gridDim.x * blockDim.x) >> 5;
    const int2 *ent2 = reinterpret_cast<const int2 *>(ent);
    for (int64_t k = warp0; k < n2; k += nwarps) {
        const int64_t row = (int64_t)__ldg(x2 + k) - row_lo;
        if (row < 0 || row >= n_rows) continue;
        const int32_t b = __ldg(ptr + row * L), e = __ldg(ptr + (row + 1) * L);
        const float *vk = V + k * ldv;
        for (int32_t i = b + lane; i < e; i += 32) {
            const int2 raw = __ldg(ent2 + i);
            const float a = __int_as_float(raw.y) * fs[(uint32_t)raw.x >> kStepShift];
            float *dst = U + (int64_t)((uint32_t)raw.x & kColMask) * ldu;
            for (int c = 0; c < t; ++c) atomicAdd(dst + c, a * __ldg(vk + c));
        }
    }
}

// Y[row, :] = sum over the row's chunks (in chunk order: deterministic) of partial[chunk, :]
__global__ void __launch_bounds__(256) long_reduce_kernel(const int32_t *__restrict__ rows,
                                                          const int32_t *__restrict__ chunk_ptr,
                                                          const float *__restrict__ partial, int64_t ldp,
                                                          float *__restrict__ Y, int64_t ldy, int32_t t,
                                                          int32_t n_long, int32_t accumulate) {
    const int64_t total = (int64_t)n_long * t;
    for (int64_t g = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; g < total;
         g += (int64_t)gridDim.x * blockDim.x) {
        const int32_t i = (int32_t)(g / t);
        const int c = (int)(g - (int64_t)i * t);
        float acc = 0.f;
        for (int32_t k = chunk_ptr[i]; k < chunk_ptr[i + 1]; ++k) acc += partial[(int64_t)k * ldp + c];
        float *dst = Y + (int64_t)rows[i] * ldy + c;
        *dst = accumulate ? *dst + acc : acc;
    }
}

// dots[i][l] = sum over the length-l entries e of row a_i of  e.val * Phi_f[b_i, col(e)],
// Phi_f[b, c] = sum_l' f[l'] * M_l'[b, c]  -- so that  sum_l f[l] * dots[i][l] = <Phi_f[a_i, :], Phi_f[b_i, :]>,
// the i-th diagonal element of K[x1, x2] (sparse_grf_kernel.py:55-57 densifies both row sets for it), and the
// columns of `dots` are what the modulator gradient of that diagonal needs.  One warp per pair: lanes take the
// entries of row a, and look each column up in the L column-sorted segments of row b (binary search).
__global__ void __launch_bounds__(256) row_dots_kernel(const int32_t *__restrict__ ptr, const GrfEntry *__restrict__ ent,
                                                       const float *__restrict__ f, int32_t L,
                                                       const int32_t *__restrict__ x1, const int32_t *__restrict__ x2,
                                                       int64_t n, int64_t row_lo, int64_t n_rows,
                                                       float *__restrict__ dots) {
    __shared__ float fs[kMaxSteps];
    if (threadIdx.x < kMaxSteps) fs[threadIdx.x] = threadIdx.x < L ? __ldg(f + threadIdx.x) : 0.f;
    __syncthreads();
    const int lane = threadIdx.x & 31;
    const int64_t warp0 = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    const int64_t n_warps = ((int64_t)gridDim.x * blockDim.x) >> 5;
    const int2 *ent2 = reinterpret_cast<const int2 *>(ent);
    for (int64_t i = warp0; i < n; i += n_warps) {
        const int64_t a = (x1 ? (int64_t)__ldg(x1 + i) : i + row_lo) - row_lo;
        const int64_t b = (x2 ? (int64_t)__ldg(x2 + i) : i + row_lo) - row_lo;
        const bool mine = a >= 0 && a < n_rows && b >= 0 && b < n_rows;   // pairs outside this shard stay zero
        for (int l = 0; l < L; ++l) {
            double acc = 0.0;
            if (mine) {
                const int32_t ab = __ldg(ptr + a * L + l), ae = __ldg(ptr + a * L + l + 1);
                for (int32_t k = ab + lane; k < ae; k += 32) {
                    const int2 ea = __ldg(ent2 + k);
                    const uint32_t col = (uint32_t)ea.x & kColMask;
                    float w = 0.f;   // Phi_f[b, col]
                    for (int m = 0; m < L; ++m) {
                        int32_t lo = __ldg(ptr + b * L + m), hi = __ldg(ptr + b * L + m + 1);
                        while (lo < hi) {
                            const int32_t mid = lo + ((hi - lo) >> 1);
                            const uint32_t c = (uint32_t)__ldg(&ent2[mid].x) & kColMask;
                            if (c < col) lo = mid + 1; else hi = mid;
                        }
                        if (lo < __ldg(ptr + b * L + m + 1)) {
                            const int2 eb = __ldg(ent2 + lo);
                            if (((uint32_t)eb.x & kColMask) == col) w = fmaf(fs[m], __int_as_float(eb.y), w);
                        }
                    }
                    acc += (double)__int_as_float(ea.y) * (double)w;
                }
            }
#pragma unroll
            for (int d = 16; d > 0; d >>= 1) acc += __shfl_xor_sync(0xffffffffu, acc, d);
            if (lane == 0) dots[i * L + l] = (float)acc;
        }
    }
}

// grad[l] += sum_k sum_c left[k, c] * (sum_{e in seg(row_k, l)} e.val * P[e.col, c])

template <int TPR, int VEC>
__global__ void __launch_bounds__(256) fgrad_blocks_kernel(const int32_t *__restrict__ ptr,
                                                           const GrfEntry *__restrict__ ent, int32_t L,
                                                           const int32_t *__restrict__ row_ids, int64_t n_tasks,
                                                           int64_t row_lo, int64_t n_rows,
                                                           const float *__restrict__ left, int64_t ldl,
                                                           const float *__restrict__ P, int64_t ldp, int32_t t,
                                                           float *__restrict__ grad) {
    __shared__ float sh[kMaxSteps];
    if (threadIdx.x < kMaxSteps) sh[threadIdx.x] = 0.f;
    __syncthreads();
    const int sub = threadIdx.x % TPR;
    const int64_t task0 = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) / TPR;
    const int64_t task_stride = ((int64_t)gridDim.x * blockDim.x) / TPR;
    for (int s = 0; s < L; ++s) {
        float g = 0.f;
        for (int64_t k = task0; k < n_tasks; k += task_stride) {
            const int64_t row = row_ids ? (int64_t)__ldg(row_ids + k) - row_lo : k;
            if (row < 0 || row >= n_rows) continue;
            const int32_t b = __ldg(ptr + row * L + s), e = __ldg(ptr + row * L + s + 1);
            for (int c0 = sub * VEC; c0 < t; c0 += TPR * VEC) {
                Vec<VEC> part;
                part.zero();
#pragma unroll 4
                for (int32_t i = b; i < e; ++i) {
                    const GrfEntry en = load_entry(ent + i);
                    Vec<VEC> x;
                    x.load(P + (int64_t)entry_col(en.col) * ldp + c0);
                    part.fma(en.val, x);
                }
                Vec<VEC> lv;
                lv.load(left + k * ldl + c0);
                g += part.dot(lv);
            }
        }
#pragma unroll
        for (int d = 16; d > 0; d >>= 1) g += __shfl_xor_sync(0xffffffffu, g, d);
        if ((threadIdx.x & 31) == 0) atomicAdd(&sh[s], g);
    }
    __syncthreads();
    if (threadIdx.x < L) atomicAdd(grad + threadIdx.x, sh[threadIdx.x]);
}

struct Shape {
    int tpr;
    int vec;
};

static Shape pick_shape(int32_t t, bool vec_ok) {
    Shape s;
    if (vec_ok) {
        s.vec = 4;
        int need = (t + 3) / 4;
        s.tpr = 1;
        while (s.tpr < need && s.tpr < 32) s.tpr <<= 1;
    } else {
        s.vec = 1;
        s.tpr = 1;
        while (s.tpr < t && s.tpr < 32) s.tpr <<= 1;
    }
    return s;
}

static inline bool aligned16(const void *p) { return ((uintptr_t)p & 15u) == 0; }

constexpr size_t kTileSmemBytes = 224 * 1024;

// Launch the tiled kernel if the windows say the matrix is banded enough; returns 1 if launched,
// 0 if the caller should use the global-gather kernel, negative on error.
static int try_launch_tiled(const int32_t *ptr, const GrfEntry *ent, const float *f, int32_t L, int64_t n_rows,
                            const int32_t *win, int32_t max_width, const float *X, int64_t ldx, float *Y,
                            int64_t ldy, int32_t t, cudaStream_t st) {
    if (!win || max_width <= 0 || t % 4 != 0 || t > 128 || n_rows < 64) return 0;
    const int ldt = (t + 3) & ~3;
    const int64_t cap_rows = (int64_t)(kTileSmemBytes / ((size_t)ldt * sizeof(float)));
    int tpr = 1;
    while (tpr * 4 < t) tpr <<= 1;
    // rows per chunk: the largest multiple of 32 such that (a) the chunk's window fits and (b) the
    // number of chunks is a multiple of the SM count (one resident CTA per SM)
    int64_t chunk = 0;
    for (int k = 1; k <= 64; ++k) {
        int64_t r = (n_rows + (int64_t)kSmCount * k - 1) / ((int64_t)kSmCount * k);
        r = (r + 31) / 32 * 32;
        if (r + max_width + 64 <= cap_rows) {
            chunk = r;
            break;
        }
    }
    if (chunk < 64 || max_width > 6 * chunk) return 0;  // too little reuse per staged byte
    const int64_t n_chunks = (n_rows + chunk - 1) / chunk;
    const int grid = (int)(n_chunks < kSmCount ? n_chunks : kSmCount);
    const size_t smem = (size_t)cap_rows * ldt * sizeof(float);
#define GRF_TILED_CASE(T)                                                                                     \
    case T: {                                                                                                 \
        auto kern = spmm_tiled_kernel<T>;                                                                     \
        GRF_CUDA_OK(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));      \
        kern<<<grid, 512, smem, st>>>(ptr, ent, f, L, n_rows, (int32_t)chunk, (const int2 *)win,             \
                                       (int32_t)cap_rows, X, ldx, Y, ldy, t);                                 \
    } break
    switch (tpr) {
        GRF_TILED_CASE(1);
        GRF_TILED_CASE(2);
        GRF_TILED_CASE(4);
        GRF_TILED_CASE(8);
        GRF_TILED_CASE(16);
        default:
            GRF_TILED_CASE(32);
    }
#undef GRF_TILED_CASE
    GRF_CUDA_OK(cudaGetLastError());
    return 1;
}

static int spmm_grid(int64_t n_tasks, int tpr) {
    const int64_t threads = n_tasks * tpr;
    int64_t g = (threads + 255) / 256;
    const int64_t cap = (int64_t)kSmCount * spmm_min_blocks(tpr);  // the resident CTAs of 256 threads per SM
    if (g > cap) g = cap;
    if (g < 1) g = 1;
    return (int)g;
}

static inline bool aligned16(const void *p);

#define GRF_DISPATCH_SHAPE(KERNEL, shape, ...)                                   \
    do {                                                                         \
        if ((shape).vec == 4) {                                                  \
            switch ((shape).tpr) {                                               \
                case 1: KERNEL<1, 4> __VA_ARGS__; break;                         \
                case 2: KERNEL<2, 4> __VA_ARGS__; break;                         \
                case 4: KERNEL<4, 4> __VA_ARGS__; break;                         \
                case 8: KERNEL<8, 4> __VA_ARGS__; break;                         \
                case 16: KERNEL<16, 4> __VA_ARGS__; break;                       \
                default: KERNEL<32, 4> __VA_ARGS__; break;                       \
            }                                                                    \
        } else {                                                                 \
            switch ((shape).tpr) {                                               \
                case 1: KERNEL<1, 1> __VA_ARGS__; break;                         \
                case 2: KERNEL<2, 1> __VA_ARGS__; break;                         \
                case 4: KERNEL<4, 1> __VA_ARGS__; break;                         \
                case 8: KERNEL<8, 1> __VA_ARGS__; break;                         \
                case 16: KERNEL<16, 1> __VA_ARGS__; break;                       \
                default: KERNEL<32, 1> __VA_ARGS__; break;                       \
            }                                                                    \
        }                                                                        \
    } while (0)

// the streaming-gather instantiations exist for the float4 shapes only (t > 2)
#define GRF_DISPATCH_SPMM(shape, stream_gather, ...)                                                \
    do {                                                                                            \
        if ((stream_gather) && (shape).vec == 4) {                                                  \
            switch ((shape).tpr) {                                                                  \
                case 1: spmm_blocks_kernel<1, 4, true> __VA_ARGS__; break;                          \
                case 2: spmm_blocks_kernel<2, 4, true> __VA_ARGS__; break;                          \
                case 4: spmm_blocks_kernel<4, 4, true> __VA_ARGS__; break;                          \
                case 8: spmm_blocks_kernel<8, 4, true> __VA_ARGS__; break;                          \
                case 16: spmm_blocks_kernel<16, 4, true> __VA_ARGS__; break;                        \
                default: spmm_blocks_kernel<32, 4, true> __VA_ARGS__; break;                        \
            }                                                                                       \
        } else {                                                                                    \
            GRF_DISPATCH_SHAPE(spmm_blocks_kernel, shape, __VA_ARGS__);                             \
        }                                                                                           \
    } while (0)

}  // namespace grf

using namespace grf;

// One half of the product on one block-CSR side: main launch (+ chunk launch and ordered
// reduction for rows longer than the split threshold).
static int launch_spmm_pass(const int32_t *ptr, const GrfEntry *ent, const float *f, int32_t L,
                            const int32_t *row_ids, int64_t n_tasks, int64_t row_lo, int64_t n_rows,
                            const GrfLongRows *lr, const float *X, int64_t ldx, float *Y, int64_t ldy, int32_t t_valid,
                            bool vec_ok, bool out_by_row, int64_t avg_row_len, int64_t x_rows, int32_t *sched,
                            bool accumulate, bool stream_gather, bool y_pad_is_scratch, cudaStream_t st) {
    // vec_ok: X rows are 16-byte aligned and padded to a multiple of 4 columns -> compute the padded
    // column count with float4 gathers.  y_pad_is_scratch: columns [t_valid, ldy) of Y are workspace (U),
    // so whole padded rows may be stored; otherwise (the caller's `out`) only the t_valid real columns are
    // written
    const bool split = lr && lr->n_long > 0 && (!row_ids || out_by_row);
    if (split) {
        GRF_REQUIRE(lr->rows && lr->chunk_ptr && lr->chunk_bounds && lr->partial && lr->ld >= t_valid,
                    "grf_phi_matvec: incomplete long-row metadata");
    }
    if (x_rows * ldx + 4 >= (1ll << 32))
        return fail(GRF_ERR_UNSUPPORTED, "grf_phi_matvec: right-hand side of %lld x %lld floats exceeds the 32-bit "
                    "element offsets of the gather kernels; split the columns", (long long)x_rows, (long long)ldx);
    if (t_valid <= 4 && avg_row_len > 64) {
        // CSR-vector path for long rows (a row subset of a W = 1000 Phi): 32 lanes per row.  Short rows
        // (config 2: 28..64 entries) are faster with one row per lane group in the kernel below.
        const bool wide = true;
        const int groups_per_cta = 256 / (wide ? 32 : 8);
        auto grid_of = [&](int64_t tasks) {
            int64_t g = (tasks + groups_per_cta - 1) / groups_per_cta;
            if (g > (int64_t)kSmCount * 8) g = (int64_t)kSmCount * 8;
            return (int)(g < 1 ? 1 : g);
        };
#define GRF_COOP(G, T, GRID, ...) spmv_coop_kernel<G, T><<<GRID, 256, 0, st>>>(__VA_ARGS__)
#define GRF_COOP_T(G, GRID, ...)                                  \
    switch (t_valid) {                                             \
        case 1: GRF_COOP(G, 1, GRID, __VA_ARGS__); break;          \
        case 2: GRF_COOP(G, 2, GRID, __VA_ARGS__); break;          \
        case 3: GRF_COOP(G, 3, GRID, __VA_ARGS__); break;          \
        default: GRF_COOP(G, 4, GRID, __VA_ARGS__); break;         \
    }
#define GRF_COOP_LAUNCH(GRID, ...)              \
    if (wide) {                                 \
        GRF_COOP_T(32, GRID, __VA_ARGS__)       \
    } else {                                    \
        GRF_COOP_T(8, GRID, __VA_ARGS__)        \
    }
        GRF_COOP_LAUNCH(grid_of(n_tasks), ptr, ent, f, L, row_ids, n_tasks, row_lo, n_rows, X, ldx, Y, ldy,
                        split ? lr->threshold : 0, nullptr, out_by_row ? 1 : 0, accumulate ? 1 : 0);
        GRF_CUDA_OK(cudaGetLastError());
        if (split) {
            GRF_COOP_LAUNCH(grid_of(lr->n_chunks), ptr, ent, f, L, nullptr, lr->n_chunks, 0, lr->n_chunks, X, ldx,
                            lr->partial, lr->ld, 0, (const int2 *)lr->chunk_bounds, 0, 0);
            GRF_CUDA_OK(cudaGetLastError());
            int64_t g = ((int64_t)lr->n_long * t_valid + 255) / 256;
            if (g > (int64_t)kSmCount * 8) g = (int64_t)kSmCount * 8;
            long_reduce_kernel<<<(int)g, 256, 0, st>>>(lr->rows, lr->chunk_ptr, lr->partial, lr->ld, Y, ldy, t_valid,
                                                       lr->n_long, accumulate ? 1 : 0);
            GRF_CUDA_OK(cudaGetLastError());
        }
#undef GRF_COOP_LAUNCH
#undef GRF_COOP_T
#undef GRF_COOP
        return GRF_OK;
    }
    const int32_t t = vec_ok ? (t_valid + 3) & ~3 : t_valid;
    const int32_t t_store = y_pad_is_scratch && ldy >= t ? t : t_valid;
    const int32_t vec_store = (ldy % 4 == 0) && aligned16(Y);
    const Shape sh = pick_shape(t, vec_ok);
    const int grid = spmm_grid(n_tasks, sh.tpr);
    GRF_DISPATCH_SPMM(sh, stream_gather,
                      <<<grid, 256, 0, st>>>(ptr, ent, f, L, row_ids, n_tasks, row_lo, n_rows, X, ldx, Y, ldy, t,
                                             t_store, vec_store, split ? lr->threshold : 0, nullptr,
                                             out_by_row ? 1 : 0, sched, accumulate ? 1 : 0));
    GRF_CUDA_OK(cudaGetLastError());
    if (split) {
        GRF_REQUIRE(lr->ld >= t, "grf_phi_matvec: long-row partial buffer narrower than the padded column count");
        const int32_t pvec = (lr->ld % 4 == 0) && aligned16(lr->partial);
        const int gridc = spmm_grid(lr->n_chunks, sh.tpr);
        GRF_DISPATCH_SPMM(sh, stream_gather,
                          <<<gridc, 256, 0, st>>>(ptr, ent, f, L, lr->chunk_order, lr->n_chunks, 0, lr->n_chunks, X,
                                                  ldx, lr->partial, lr->ld, t, t, pvec, 0,
                                                  (const int2 *)lr->chunk_bounds, 0, sched, 0));
        GRF_CUDA_OK(cudaGetLastError());
        int64_t g = ((int64_t)lr->n_long * t + 255) / 256;
        if (g > (int64_t)kSmCount * 8) g = (int64_t)kSmCount * 8;
        long_reduce_kernel<<<(int)g, 256, 0, st>>>(lr->rows, lr->chunk_ptr, lr->partial, lr->ld, Y, ldy, t_store,
                                                   lr->n_long, accumulate ? 1 : 0);
        GRF_CUDA_OK(cudaGetLastError());
    }
    return GRF_OK;
}

extern "C" int grf_phi_matvec(const GrfPhi *phi, const float *f, const int32_t *x1, int64_t n1, const int32_t *x2,
                              int64_t n2, const float *v, int64_t ldv, float *out, int64_t ldo, float *u, int64_t ldu,
                              float *vfull, int32_t t, int32_t which, void *stream) {
    GRF_ON_STREAM_DEVICE(stream, u);
    GRF_REQUIRE(phi && f, "grf_phi_matvec: null phi/f");
    GRF_REQUIRE(t >= 1, "grf_phi_matvec: t must be >= 1");
    GRF_REQUIRE((which & 3) >= 1 && which <= 63, "grf_phi_matvec: which must be 1, 2 or 3 (+4, +8, +16, +32 flags)");
    GRF_REQUIRE(phi->n_steps >= 1 && phi->n_steps <= kMaxSteps, "grf_phi_matvec: n_steps out of range");
    GRF_REQUIRE(phi->n_cols <= (1ll << kStepShift) && phi->n_rows <= (1ll << kStepShift),
                "grf_phi_matvec: more than 2^27 rows or columns per GPU");
    GRF_REQUIRE(u && ldu >= t, "grf_phi_matvec: U workspace missing or ldu < t");
    GRF_REQUIRE(x1 || n1 == phi->n_rows, "grf_phi_matvec: n1 must equal n_rows when x1 is NULL");
    GRF_REQUIRE(x2 || n2 == phi->n_rows, "grf_phi_matvec: n2 must equal n_rows when x2 is NULL");
    cudaStream_t st = (cudaStream_t)stream;
    const int32_t L = phi->n_steps;
    const int64_t avg_len = phi->nnz > 0 && phi->n_rows > 0 ? phi->nnz / phi->n_rows : 0;  // entries per row of Phi
    const int tile_mode = (which >> 2) & 1;  // +4: never use the shared-memory-tiled kernel
    const bool x2_unique = (which >> 3) & 1;  // +8: x2 has no repeated ids and vfull was zeroed once
    const bool accumulate = (which >> 4) & 1;  // +16: U += (later row blocks of a block-wise Phi^T)
    const bool stream_gather = (which >> 5) & 1;  // +32: L1::no_allocate gathers
    which &= 3;

    if (which & 1) {
        GRF_REQUIRE(v && ldv >= t, "grf_phi_matvec: V missing or ldv < t");
        GRF_REQUIRE(phi->tblk_ptr, "grf_phi_matvec: Phi^T blocks missing");
        const float *src = v;
        int64_t lds = ldv;
        const bool scatter_half = x2 && phi->blk_ptr && n2 * 16 < phi->n_rows;
        if (scatter_half) {
            // small row subset: scatter from the selected rows of Phi instead of a pass over Phi^T
            if (!accumulate) GRF_CUDA_OK(cudaMemsetAsync(u, 0, (size_t)phi->n_cols * ldu * sizeof(float), st));
            if (n2 > 0) {
                int64_t g = (n2 + 7) / 8;
                if (g > (int64_t)kSmCount * 8) g = (int64_t)kSmCount * 8;
                spmm_scatter_kernel<<<(int)g, 256, 0, st>>>(phi->blk_ptr, phi->entries, f, L, x2, n2, phi->row_lo,
                                                            phi->n_rows, v, ldv, u, ldu, t);
                GRF_CUDA_OK(cudaGetLastError());
            }
        } else if (x2) {
            GRF_REQUIRE(vfull, "grf_phi_matvec: vfull workspace needed when x2 is given");
            // x2_unique: the caller guarantees no repeated ids and a vfull that was zeroed once; rows
            // outside x2 then stay zero across calls and the scatter needs neither memset nor atomics
            if (!x2_unique) GRF_CUDA_OK(cudaMemsetAsync(vfull, 0, (size_t)phi->n_rows * ldu * sizeof(float), st));
            if (n2 > 0 && phi->n_rows > 0) {
                int64_t g = (n2 * t + 255) / 256;
                if (g > (int64_t)kSmCount * 16) g = (int64_t)kSmCount * 16;
                if (x2_unique)
                    scatter_rows_unique_kernel<<<(int)g, 256, 0, st>>>(x2, n2, phi->row_lo, phi->n_rows, v, ldv,
                                                                      vfull, ldu, t);
                else
                    scatter_rows_kernel<<<(int)g, 256, 0, st>>>(x2, n2, phi->row_lo, phi->n_rows, v, ldv, vfull,
                                                               ldu, t);
                GRF_CUDA_OK(cudaGetLastError());
            }
            src = vfull;
            lds = ldu;
        } else if (vfull && phi->n_rows > 0 && t > 2 && (ldv % 4 != 0 || !aligned16(v)) && ldu % 4 == 0) {
            // V is not laid out for 16-byte gathers (e.g. t = 17): stage it in the padded buffer
            int64_t g = (phi->n_rows * t + 255) / 256;
            if (g > (int64_t)kSmCount * 16) g = (int64_t)kSmCount * 16;
            pad_copy_kernel<<<(int)g, 256, 0, st>>>(v, ldv, vfull, ldu, phi->n_rows, t);
            GRF_CUDA_OK(cudaGetLastError());
            src = vfull;
            lds = ldu;
        }
        if (scatter_half) {
            // done above
        } else if (phi->n_cols > 0 && phi->n_rows == 0) {
            // empty shard: its partial sum is zero (and there is no row of V to read)
            if (!accumulate)
                GRF_CUDA_OK(cudaMemset2DAsync(u, (size_t)ldu * sizeof(float), 0, (size_t)t * sizeof(float),
                                              (size_t)phi->n_cols, st));
        } else if (phi->n_cols > 0) {
            const int32_t t4 = (t + 3) & ~3;
            // one or two columns: scalar lanes beat float4 gathers that are 3/4 padding
            const bool vec_ok = t > 2 && (lds % 4 == 0) && (ldu % 4 == 0) && lds >= t4 && ldu >= t4 && aligned16(src) &&
                                aligned16(u);
            int tiled = 0;
            if (vec_ok && t % 4 == 0 && !(tile_mode & 1) && !accumulate) {
                tiled = try_launch_tiled(phi->tblk_ptr, phi->tentries, f, L, phi->n_cols, phi->twin,
                                         phi->twin_max_width, src, lds, u, ldu, t, st);
                if (tiled < 0) return tiled;
            }
            if (!tiled) {
                int rc;
                if (phi->tcols) {
                    // only the listed columns (those this shard touches, in any order); the others are zero
                    if (phi->n_tcols < phi->n_cols && !accumulate)
                        GRF_CUDA_OK(cudaMemsetAsync(u, 0, (size_t)phi->n_cols * ldu * sizeof(float), st));
                    rc = phi->n_tcols == 0
                             ? GRF_OK
                             : launch_spmm_pass(phi->tblk_ptr, phi->tentries, f, L, phi->tcols, phi->n_tcols, 0,
                                                phi->n_cols, phi->long_t, src, lds, u, ldu, t, vec_ok, true, avg_len, phi->n_rows, phi->sched,
                                                accumulate, stream_gather, true, st);
                } else {
                    rc = launch_spmm_pass(phi->tblk_ptr, phi->tentries, f, L, nullptr, phi->n_cols, 0, phi->n_cols,
                                          phi->long_t, src, lds, u, ldu, t, vec_ok, false, avg_len, phi->n_rows, phi->sched,
                                          accumulate, stream_gather, true, st);
                }
                if (rc != GRF_OK) return rc;
            }
        }
    }
    if ((which & 2) && n1 > 0) {
        GRF_REQUIRE(out && ldo >= t, "grf_phi_matvec: out missing or ldo < t");
        GRF_REQUIRE(phi->blk_ptr, "grf_phi_matvec: Phi blocks missing");
        const int32_t t4 = (t + 3) & ~3;
        const bool vec_ok = t > 2 && (ldu % 4 == 0) && ldu >= t4 && aligned16(u);   // gathers come from U
        int tiled = 0;
        if (vec_ok && t % 4 == 0 && (ldo % 4 == 0) && aligned16(out) && !x1 && !(tile_mode & 1)) {
            tiled = try_launch_tiled(phi->blk_ptr, phi->entries, f, L, phi->n_rows, phi->win, phi->win_max_width, u,
                                     ldu, out, ldo, t, st);
            if (tiled < 0) return tiled;
        }
        if (!tiled) {
            const int rc = launch_spmm_pass(phi->blk_ptr, phi->entries, f, L, x1, n1, phi->row_lo, phi->n_rows,
                                            phi->long_fwd, u, ldu, out, ldo, t, vec_ok, false, avg_len, phi->n_cols, phi->sched,
                                            false, stream_gather, false, st);
            if (rc != GRF_OK) return rc;
        }
    }
    return GRF_OK;
}

extern "C" int grf_phi_fgrad(const GrfPhi *phi, const int32_t *x, int64_t n, const float *left, int64_t ldl,
                             const float *p, int64_t ldp, int32_t t, float *grad, void *stream) {
    GRF_ON_STREAM_DEVICE(stream, grad);
    GRF_REQUIRE(phi && left && p && grad, "grf_phi_fgrad: null argument");
    GRF_REQUIRE(t >= 1 && ldl >= t && ldp >= t, "grf_phi_fgrad: bad t / leading dimensions");
    GRF_REQUIRE(phi->n_steps >= 1 && phi->n_steps <= kMaxSteps, "grf_phi_fgrad: n_steps out of range");
    GRF_REQUIRE(x || n == phi->n_rows, "grf_phi_fgrad: n must equal n_rows when x is NULL");
    if (n == 0) return GRF_OK;
    GRF_REQUIRE(phi->blk_ptr, "grf_phi_fgrad: Phi blocks missing");
    const bool vec_ok = (t % 4 == 0) && (ldl % 4 == 0) && (ldp % 4 == 0) && aligned16(left) && aligned16(p);
    const Shape sh = pick_shape(t, vec_ok);
    int grid = spmm_grid(n, sh.tpr);
    if (grid > kSmCount * 4) grid = kSmCount * 4;
    GRF_DISPATCH_SHAPE(fgrad_blocks_kernel, sh,
                       <<<grid, 256, 0, (cudaStream_t)stream>>>(phi->blk_ptr, phi->entries, phi->n_steps, x, n,
                                                                phi->row_lo, phi->n_rows, left, ldl, p, ldp, t, grad));
    return check_cuda(cudaGetLastError(), "fgrad_blocks_kernel launch");
}

extern "C" int grf_phi_row_dots(const GrfPhi *phi, const float *f, const int32_t *x1, const int32_t *x2, int64_t n,
                                float *dots, void *stream) {
    GRF_ON_STREAM_DEVICE(stream, dots);
    GRF_REQUIRE(phi && f && dots, "grf_phi_row_dots: null argument");
    GRF_REQUIRE(phi->n_steps >= 1 && phi->n_steps <= kMaxSteps, "grf_phi_row_dots: n_steps out of range");
    GRF_REQUIRE(n >= 0, "grf_phi_row_dots: negative n");
    GRF_REQUIRE((x1 && x2) || n == phi->n_rows, "grf_phi_row_dots: n must equal n_rows when an index list is NULL");
    if (n == 0) return GRF_OK;
    GRF_REQUIRE(phi->blk_ptr, "grf_phi_row_dots: Phi blocks missing");
    int64_t g = (n + 7) / 8;
    if (g > (int64_t)kSmCount * 16) g = (int64_t)kSmCount * 16;
    row_dots_kernel<<<(int)g, 256, 0, (cudaStream_t)stream>>>(phi->blk_ptr, phi->entries, f, phi->n_steps, x1, x2, n,
                                                              phi->row_lo, phi->n_rows, dots);
    return check_cuda(cudaGetLastError(), "row_dots_kernel launch");
}

extern "C" int grf_block_windows(const int32_t *blk_ptr, const GrfEntry *entries, int64_t n_rows, int32_t n_steps,
                                 int32_t *win, int32_t *max_width, void *stream) {
    GRF_ON_STREAM_DEVICE(stream, max_width);
    GRF_REQUIRE(n_rows >= 0 && n_steps >= 1, "grf_block_windows: bad shape");
    GRF_REQUIRE(max_width, "grf_block_windows: null max_width");
    cudaStream_t st = (cudaStream_t)stream;
    GRF_CUDA_OK(cudaMemsetAsync(max_width, 0, sizeof(int32_t), st));
    if (n_rows == 0) return GRF_OK;
    GRF_REQUIRE(blk_ptr && win, "grf_block_windows: null buffer");
    const int64_t n_groups = (n_rows + 31) / 32;
    int64_t g = (n_groups + 7) / 8;
    if (g > (int64_t)kSmCount * 16) g = (int64_t)kSmCount * 16;
    block_windows_kernel<<<(int)g, 256, 0, st>>>(blk_ptr, entries, n_rows, n_steps, (int2 *)win, max_width);
    return check_cuda(cudaGetLastError(), "block_windows_kernel launch");
}
