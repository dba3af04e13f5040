// Alias tables for weight-proportional neighbour draws (grf_alias_records; definitions at GrfAliasEdge in
// include/grf_b200.h).  No reference counterpart: the reference draws neighbours uniformly.
//
// One thread group builds one row: a warp per row of <= kLongRow entries, a CTA per longer row (the hub row of
// config 4 has 175 304 entries).  A row of <= 32 entries is built in registers (alias_row_small below: the same
// arithmetic, every pass a shuffle).  Longer rows take five passes, the output region doubling as scratch:
//   1. S: lanes 0..31 of the first warp add the lane-strided partial sums in index order, then the fixed tree
//      (one warp's shuffle reduction) -- the definition's order, 32-way parallel;
//   2. masses m_k = floor((a_k * D) / S) into out[k].scaled (as uint64), their sum and the largest (lowest
//      index) by group reductions; the deficit goes to that one entry;
//   3. compaction in index order: tile by tile, each thread takes IPT consecutive entries, one group scan per
//      tile.  Light item r (m < 2^32) leaves {Lx_r = deficits (2^32 - m) of the lights before it, index} in
//      out[r].{scaled_alias, col_alias}; heavy item q leaves {Hx_q = excesses (m - 2^32) of the heavies
//      before it, index} in out[nL + q];
//   4. the sweep as searches: the sequential sweep consumes the heavies' excesses in order as a line, so light
//      r is aliased to the heavy q whose stretch [Hx_q, Hx_{q+1}) holds Lx_r, and heavy q runs out at the
//      first light boundary P = min {Lx_t (or the total) >= Hx_{q+1}}: thr_q = 2^32 - (P - Hx_{q+1}), alias
//      q + 1, full when P = Hx_{q+1} or q is the last heavy.  Results (alias index, thr) go to
//      out[k].{col, thr}, fields the scratch does not use;
//   5. the records themselves, each thread its own entries.
// Every value after the masses is an integer function of the row: bit-identical to the sequential sweep of
// oracle/grf_oracle_weighted.c, whatever the group size.

#include <limits.h>

#include "grf_common.cuh"

namespace grf {
namespace {

constexpr int kLongRow = 2048;  // longer rows take a CTA
constexpr int kCtaThreads = 256;
constexpr int kIpt = 8;  // consecutive entries per thread per compaction tile
constexpr unsigned long long kT = 1ull << 32;

template <bool kBlock>
__device__ __forceinline__ void gsync() {
    if (kBlock)
        __syncthreads();
    else
        __syncwarp();
}

// exclusive scan of one uint64 per thread over the group; `total` = group sum
template <bool kBlock>
__device__ __forceinline__ unsigned long long gscan(unsigned long long v, unsigned long long *scratch,
                                                    unsigned long long &total) {
    const int lane = threadIdx.x & 31;
    unsigned long long incl = v;
#pragma unroll
    for (int d = 1; d < 32; d <<= 1) {
        const unsigned long long n = __shfl_up_sync(0xffffffffu, incl, d);
        if (lane >= d) incl += n;
    }
    if (!kBlock) {
        total = __shfl_sync(0xffffffffu, incl, 31);
        return incl - v;
    }
    const int warp = threadIdx.x >> 5, nwarps = blockDim.x >> 5;
    if (lane == 31) scratch[warp] = incl;
    __syncthreads();
    unsigned long long before = 0, all = 0;
    for (int i = 0; i < nwarps; ++i) {
        const unsigned long long s = scratch[i];
        if (i < warp) before += s;
        all += s;
    }
    __syncthreads();
    total = all;
    return before + incl - v;
}

// the largest m over the group, lowest index among ties
template <bool kBlock>
__device__ __forceinline__ void gargmax(unsigned long long &m, int &idx, unsigned long long *scratch) {
#pragma unroll
    for (int d = 16; d > 0; d >>= 1) {
        const unsigned long long om = __shfl_xor_sync(0xffffffffu, m, d);
        const int oi = __shfl_xor_sync(0xffffffffu, idx, d);
        if (om > m || (om == m && oi < idx)) {
            m = om;
            idx = oi;
        }
    }
    if (!kBlock) return;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, nwarps = blockDim.x >> 5;
    if (lane == 0) {
        scratch[2 * warp] = m;
        scratch[2 * warp + 1] = (unsigned long long)(unsigned)idx;
    }
    __syncthreads();
    for (int i = 0; i < nwarps; ++i) {
        const unsigned long long om = scratch[2 * i];
        const int oi = (int)scratch[2 * i + 1];
        if (om > m || (om == m && oi < idx)) {
            m = om;
            idx = oi;
        }
    }
    __syncthreads();
}

__device__ __forceinline__ unsigned long long as_u64(double x) { return (unsigned long long)__double_as_longlong(x); }
__device__ __forceinline__ double as_f64(unsigned long long x) { return __longlong_as_double((long long)x); }
__device__ __forceinline__ void st_u64(double *p, unsigned long long x) { *p = as_f64(x); }  // scratch in a double field

// first position in [lo, hi) of the compacted prefixes (out[rs + t].scaled_alias) whose value is > x (kUpper)
// or >= x (!kUpper); plain loads: this group wrote them
template <bool kUpper>
__device__ __forceinline__ int search(const GrfAliasEdge *o, int lo, int hi, unsigned long long x) {
    while (lo < hi) {
        const int mid = (lo + hi) >> 1;
        const unsigned long long v = as_u64(o[mid].scaled_alias);
        if (kUpper ? v <= x : v < x)
            lo = mid + 1;
        else
            hi = mid;
    }
    return lo;
}

template <bool kBlock>
__device__ void alias_row(const int32_t *__restrict__ col, const double *__restrict__ val, int32_t rs, int32_t d,
                          double one_minus_p, GrfAliasEdge *out, unsigned long long *scratch, double *s_bcast) {
    const int GS = kBlock ? (int)blockDim.x : 32;
    const int tg = kBlock ? (int)threadIdx.x : (int)(threadIdx.x & 31);
    GrfAliasEdge *o = out + rs;
    const double *w = val + rs;

    // ---- 1. S ----
    double S;
    if (!kBlock || tg < 32) {
        double s = 0.0;
        int32_t k = tg;
        for (; k + 32 * 7 < d; k += 32 * 8) {  // eight loads in flight, added in index order
            double a[8];
#pragma unroll
            for (int u = 0; u < 8; ++u) a[u] = fabs(w[k + 32 * u]);
#pragma unroll
            for (int u = 0; u < 8; ++u) s = __dadd_rn(s, a[u]);
        }
        for (; k < d; k += 32) s = __dadd_rn(s, fabs(w[k]));
#pragma unroll
        for (int h = 16; h > 0; h >>= 1) {
            const double o2 = __shfl_down_sync(0xffffffffu, s, h);
            if (tg < h) s = __dadd_rn(s, o2);
        }
        S = __shfl_sync(0xffffffffu, s, 0);
        if (kBlock && tg == 0) *s_bcast = S;
    }
    if (kBlock) {
        __syncthreads();
        S = *s_bcast;
        __syncthreads();
    }

    // ---- 2. masses, their sum, the largest ----
    const bool live = S > 0.0;
    const double D = (double)d * 4294967296.0;
    unsigned long long msum = 0, mbig = 0, my_light = 0;
    int ibig = INT_MAX;
    for (int32_t k = tg; k < d; k += GS) {
        const unsigned long long m = live ? (unsigned long long)floor(__ddiv_rn(__dmul_rn(fabs(w[k]), D), S)) : kT;
        st_u64(&o[k].scaled, m);
        msum += m;
        my_light += m < kT;
        if (m > mbig || (m == mbig && k < ibig)) {
            mbig = m;
            ibig = k;
        }
    }
    unsigned long long all, n_light;
    gscan<kBlock>(msum, scratch, all);
    gscan<kBlock>(my_light, scratch, n_light);
    gargmax<kBlock>(mbig, ibig, scratch);
    // the deficit moves the largest mass; every thread knows the light count after the move
    const unsigned long long mnew =
        live ? (unsigned long long)((long long)mbig + ((long long)((unsigned long long)d * kT) - (long long)all)) : mbig;
    const int nl_all = (int)n_light - (mbig < kT) + (mnew < kT);
    gsync<kBlock>();  // every mass is stored
    if (tg == 0 && live) st_u64(&o[ibig].scaled, mnew);
    gsync<kBlock>();

    // ---- 3. compaction: lights and heavies in index order with exclusive prefix sums ----
    unsigned long long lsum = 0, hsum = 0;  // running totals of the tiles before
    int nl = 0, nh = 0;
    for (int32_t t0 = 0; t0 < d; t0 += GS * kIpt) {
        const int32_t k0 = t0 + tg * kIpt;
        unsigned long long m[kIpt];
        unsigned long long my_l = 0, my_h = 0;
        int my_nl = 0, my_nh = 0;
#pragma unroll
        for (int i = 0; i < kIpt; ++i) {
            m[i] = k0 + i < d ? as_u64(o[k0 + i].scaled) : kT;
            if (m[i] < kT) {
                my_l += kT - m[i];
                ++my_nl;
            } else if (m[i] > kT) {
                my_h += m[i] - kT;
                ++my_nh;
            }
        }
        unsigned long long tl, th, tc;
        unsigned long long pl = gscan<kBlock>(my_l, scratch, tl);
        unsigned long long ph = gscan<kBlock>(my_h, scratch, th);
        const unsigned long long pc = gscan<kBlock>((unsigned long long)my_nl | ((unsigned long long)my_nh << 32),
                                                    scratch, tc);
        // the compacted records live in fields the masses do not use: no hazard with the reads above
        int rl = nl + (int)(uint32_t)pc, rh = nl_all + nh + (int)(pc >> 32);
        pl += lsum;
        ph += hsum;
#pragma unroll
        for (int i = 0; i < kIpt; ++i) {
            if (m[i] < kT) {
                st_u64(&o[rl].scaled_alias, pl);
                o[rl].col_alias = k0 + i;
                pl += kT - m[i];
                ++rl;
            } else if (m[i] > kT) {
                st_u64(&o[rh].scaled_alias, ph);
                o[rh].col_alias = k0 + i;
                ph += m[i] - kT;
                ++rh;
            }
        }
        lsum += tl;
        hsum += th;
        nl += (int)(uint32_t)tc;
        nh += (int)(tc >> 32);
    }
    gsync<kBlock>();

    // ---- 4. the sweep as searches ----
    const unsigned long long total = lsum;  // == hsum: the masses add up to d * 2^32
    for (int32_t k = tg; k < d; k += GS)
        if (as_u64(o[k].scaled) == kT) {  // full bucket (S = 0 rows: all of them)
            o[k].col = k;
            o[k].thr = 0xffffffffu;
        }
    for (int r = tg; r < nl; r += GS) {
        const unsigned long long lx = as_u64(o[r].scaled_alias);
        const int k = o[r].col_alias;
        const int q = search<true>(o + nl, 1, nh, lx) - 1;  // heavies q' >= 1 with Hx_q' <= Lx_r
        o[k].col = o[nl + q].col_alias;
        o[k].thr = (uint32_t)as_u64(o[k].scaled);
    }
    for (int q = tg; q < nh; q += GS) {
        const int k = o[nl + q].col_alias;
        uint32_t thr = 0xffffffffu;
        int32_t alias = k;
        if (q + 1 < nh) {
            const unsigned long long hnext = as_u64(o[nl + q + 1].scaled_alias);
            const int t = search<false>(o, 0, nl, hnext);
            const unsigned long long P = t < nl ? as_u64(o[t].scaled_alias) : total;
            if (P > hnext) {
                thr = (uint32_t)(kT - (P - hnext));
                alias = o[nl + q + 1].col_alias;
            }
        }
        o[k].col = alias;
        o[k].thr = thr;
    }
    gsync<kBlock>();

    // ---- 5. the records ----
    const double q = live ? __ddiv_rn(S, one_minus_p) : 0.0;
    for (int32_t k = tg; k < d; k += GS) {
        const int32_t a = o[k].col;
        GrfAliasEdge e;
        e.scaled = live ? (w[k] < 0.0 ? -q : q) : 0.0;
        e.scaled_alias = live ? (w[a] < 0.0 ? -q : q) : 0.0;
        e.col = col[rs + k];
        e.col_alias = col[rs + a];
        e.thr = o[k].thr;
        e.pad = 0;
        o[k] = e;
    }
    gsync<kBlock>();  // the next row of this group may use shared scratch
}

// A row of <= 32 entries (most rows of a sparse graph): lane k holds entry k and every pass of alias_row is a
// shuffle -- the same arithmetic in the same order, nothing parked in memory.  Heavy items have strictly increasing
// Hx in index order, so light r's alias (the last heavy with Hx <= Lx_r) and heavy q's boundary P (the smallest
// Lx >= Hx_{q+1}) are one 32-step scan over the lanes each.
__device__ void alias_row_small(const int32_t *__restrict__ col, const double *__restrict__ val, int32_t rs,
                                int32_t d, double one_minus_p, GrfAliasEdge *out) {
    const int lane = threadIdx.x & 31;
    const bool in = lane < d;
    const double wv = in ? val[rs + lane] : 0.0;
    const int32_t cv = in ? col[rs + lane] : 0;
    // S: s_lane = 0.0 + |w_lane| (exact), then the fixed tree
    double s = fabs(wv);
#pragma unroll
    for (int h = 16; h > 0; h >>= 1) {
        const double o2 = __shfl_down_sync(0xffffffffu, s, h);
        if (lane < h) s = __dadd_rn(s, o2);
    }
    const double S = __shfl_sync(0xffffffffu, s, 0);
    const bool live = S > 0.0;
    const double D = (double)d * 4294967296.0;
    unsigned long long m = in ? (live ? (unsigned long long)floor(__ddiv_rn(__dmul_rn(fabs(wv), D), S)) : kT) : 0;
    unsigned long long msum = m, mbig = m;
    int ibig = in ? lane : INT_MAX;
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
        msum += __shfl_xor_sync(0xffffffffu, msum, o);
        const unsigned long long om = __shfl_xor_sync(0xffffffffu, mbig, o);
        const int oi = __shfl_xor_sync(0xffffffffu, ibig, o);
        if (om > mbig || (om == mbig && oi < ibig)) {
            mbig = om;
            ibig = oi;
        }
    }
    if (live && lane == ibig) m = (unsigned long long)((long long)m + ((long long)((unsigned long long)d * kT) - (long long)msum));
    if (!in) m = kT;
    const bool light = m < kT, heavy = m > kT;
    // exclusive prefix sums of the light deficits and heavy excesses in index order
    unsigned long long lx = light ? kT - m : 0, hx = heavy ? m - kT : 0;
    const unsigned long long dl = lx, dh = hx;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
        const unsigned long long a = __shfl_up_sync(0xffffffffu, lx, o), b = __shfl_up_sync(0xffffffffu, hx, o);
        if (lane >= o) {
            lx += a;
            hx += b;
        }
    }
    const unsigned long long total = __shfl_sync(0xffffffffu, lx, 31);
    lx -= dl;
    hx -= dh;
    const uint32_t bl = __ballot_sync(0xffffffffu, light), bh = __ballot_sync(0xffffffffu, heavy);
    const uint32_t above = (uint32_t)(bh & ~((2ull << lane) - 1));  // heavies after this lane
    const int nj = above ? __ffs(above) - 1 : 0;                    // the next heavy item
    const unsigned long long hnext = __shfl_sync(0xffffffffu, hx, nj);
    int light_alias = 0;
    unsigned long long P = total;
    for (int j = 0; j < 32; ++j) {
        const unsigned long long hj = __shfl_sync(0xffffffffu, hx, j), lj = __shfl_sync(0xffffffffu, lx, j);
        if (((bh >> j) & 1u) && hj <= lx) light_alias = j;
        if (((bl >> j) & 1u) && lj >= hnext && lj < P) P = lj;
    }
    uint32_t thr = 0xffffffffu;
    int alias = lane;
    if (light) {
        thr = (uint32_t)m;
        alias = light_alias;
    } else if (heavy && above && P > hnext) {
        thr = (uint32_t)(kT - (P - hnext));
        alias = nj;
    }
    const int neg = wv < 0.0;
    const int neg_alias = __shfl_sync(0xffffffffu, neg, alias);
    const int32_t col_alias = __shfl_sync(0xffffffffu, cv, alias);
    if (!in) return;
    const double q = live ? __ddiv_rn(S, one_minus_p) : 0.0;
    GrfAliasEdge e;
    e.scaled = live ? (neg ? -q : q) : 0.0;
    e.scaled_alias = live ? (neg_alias ? -q : q) : 0.0;
    e.col = cv;
    e.col_alias = col_alias;
    e.thr = thr;
    e.pad = 0;
    out[rs + lane] = e;
}

__global__ void __launch_bounds__(256) alias_rows_warp(const int32_t *__restrict__ row_ptr,
                                                       const int32_t *__restrict__ col,
                                                       const double *__restrict__ val, int64_t n_nodes,
                                                       double one_minus_p, GrfAliasEdge *out) {
    const int64_t warp0 = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    const int64_t nwarps = ((int64_t)gridDim.x * blockDim.x) >> 5;
    for (int64_t r = warp0; r < n_nodes; r += nwarps) {
        const int32_t b = row_ptr[r], d = row_ptr[r + 1] - b;
        if (d == 0 || d > kLongRow) continue;
        if (d <= 32)
            alias_row_small(col, val, b, d, one_minus_p, out);
        else
            alias_row<false>(col, val, b, d, one_minus_p, out, nullptr, nullptr);
    }
}

__global__ void __launch_bounds__(kCtaThreads) alias_rows_cta(const int32_t *__restrict__ row_ptr,
                                                              const int32_t *__restrict__ col,
                                                              const double *__restrict__ val, int64_t n_nodes,
                                                              double one_minus_p, GrfAliasEdge *out) {
    __shared__ unsigned long long scratch[2 * (kCtaThreads / 32)];
    __shared__ double s_bcast;
    __shared__ int32_t longs[kCtaThreads];
    __shared__ int n_long;
    // row r belongs to CTA r mod gridDim.x (R-MAT numbers its hubs first: contiguous chunks would hand most hub
    // rows to one CTA); per round a CTA collects the long rows among blockDim.x of its own, then builds them one
    // at a time with the whole CTA
    for (int64_t base = 0; base < n_nodes; base += (int64_t)gridDim.x * blockDim.x) {
        if (threadIdx.x == 0) n_long = 0;
        __syncthreads();
        const int64_t r = base + (int64_t)threadIdx.x * gridDim.x + blockIdx.x;
        if (r < n_nodes && row_ptr[r + 1] - row_ptr[r] > kLongRow) longs[atomicAdd(&n_long, 1)] = (int32_t)r;
        __syncthreads();
        const int nlong = n_long;
        for (int i = 0; i < nlong; ++i) {
            const int32_t rr = longs[i];
            const int32_t b = row_ptr[rr], d = row_ptr[rr + 1] - b;
            alias_row<true>(col, val, b, d, one_minus_p, out, scratch, &s_bcast);
        }
        __syncthreads();
    }
}

}  // namespace
}  // namespace grf

extern "C" int grf_alias_records(const GrfGraph *graph, double p_halt, GrfAliasEdge *out, void *stream) {
    GRF_ON_STREAM_DEVICE(stream, out);
    using namespace grf;
    GRF_REQUIRE(graph, "grf_alias_records: null graph");
    GRF_REQUIRE(p_halt >= 0.0 && p_halt <= 1.0, "grf_alias_records: p_halt must be in [0, 1]");
    GRF_REQUIRE(graph->n_nodes >= 0 && graph->n_nodes < (1ll << 31), "grf_alias_records: n_nodes out of range");
    GRF_REQUIRE(graph->nnz >= 0 && graph->nnz < (1ll << 31), "grf_alias_records: nnz out of range");
    if (graph->n_nodes == 0 || graph->nnz == 0) return GRF_OK;
    GRF_REQUIRE(graph->row_ptr && graph->col_idx && graph->val && out, "grf_alias_records: null buffer");
    cudaStream_t st = (cudaStream_t)stream;
    int64_t g = (graph->n_nodes + 7) / 8;
    if (g > (int64_t)kSmCount * 32) g = (int64_t)kSmCount * 32;
    alias_rows_warp<<<(int)g, 256, 0, st>>>(graph->row_ptr, graph->col_idx, graph->val, graph->n_nodes,
                                            1.0 - p_halt, out);
    GRF_CUDA_OK(cudaGetLastError());
    int64_t gc = (graph->n_nodes + kCtaThreads - 1) / kCtaThreads;
    if (gc > (int64_t)kSmCount * 8) gc = (int64_t)kSmCount * 8;
    alias_rows_cta<<<(int)gc, kCtaThreads, 0, st>>>(graph->row_ptr, graph->col_idx, graph->val, graph->n_nodes,
                                                   1.0 - p_halt, out);
    return check_cuda(cudaGetLastError(), "alias_rows launch");
}
