// GRF walker + per-start-node merge (K1 + the dict half of K2 in SURVEY.md 2a).
//
// Replaces the reference's CPython walk loop
//   efficient_graph_gp_sparse/random_walk_samplers_sparse/sparse_sampler.py:36-54
//   efficient_graph_gp/random_walk_samplers/sampler.py:40-59, :163-184
// and its defaultdict accumulation / merge (:42, :110-114).
//
// One *group* (a warp, or a whole CTA when W is large) owns one start node at a
// time.  Phase 1: every lane runs walks w = lane, lane+G, ... of that node:
// CSR row_ptr pair -> halting draw -> neighbour draw -> (col, val) gather, the
// load update deg*w/(1-p) applied in registers in float64, and the visit
// (node, load) of every length >= 1 parked in shared memory.  Phase 2: per
// length, the <= W visits are bitonic-sorted by (node, walk) -- in registers
// with warp shuffles when a warp owns the node, in shared memory when a CTA
// does -- and, per distinct node, the loads are added *in walk order* into a double
// that starts at 0.0 -- exactly the order in which the reference's
// defaultdict(float) accumulates them, so the sums are bit-identical when both
// sides see the same draws.  The merged (column-sorted) per-length segments go
// to the row's staging region; grf_compact_* turns staging into CSR.
//
// Draw sources: Philox4x32-10 keyed by the seed with counter (walk id, step / 2)
// -- one block serves two steps: words (0, 1) halt / pick the even step, words
// (2, 3) the odd one; independent of how start nodes are sharded over GPUs --
// or a replayed trace of the reference's own PCG64 draws.
//
// Roofline: per executed walk-step the algorithmic traffic is row_ptr pair 8 B
// + col 4 B + val 8 B + staging write 12 B/(merged entry); three dependent
// random 32-B sectors per step => latency / sector bound, not bandwidth bound.

#include <limits.h>
#include <stdlib.h>

#include "grf_common.cuh"

namespace grf {

struct WalkParams {
    const int32_t *row_ptr;
    const int32_t *col_idx;
    const double *val;
    const GrfEdge *edges;
    int64_t start_lo;
    int64_t n_local;
    int32_t W, L, Wp, wbits;
    double p_halt, one_minus_p;
    unsigned long long halt_thr;
    uint32_t k0, k1;
    int32_t draw_mode, load_mode;
    const double *trace_u;
    const int32_t *trace_k;
    int64_t stride;
    int32_t *stage_col;
    double *stage_sum;
    int32_t *row_cnt;
    unsigned long long *visits;
    uint32_t group_bytes, loads_bytes, nodes_bytes, sorted_bytes;
    int32_t *col_counts;  // optional [n_nodes][L]: entries per (column, length), for the Phi^T offsets
    long long trace_base;  // replay: trace element 0 belongs to this walk id
    GrfEntry *stage_ent;   // optional: finished Phi entries instead of (stage_col, stage_sum)
    int32_t scale_mode;
    double recip_w, w_as_double;
};

// L2 eviction hints (createpolicy + ld.global.L2::cache_hint).  On a graph that does not fit L2 (config 4:
// 0.6 GB of columns, 1.2 GB of load factors) every gathered edge is used once and streams through; the
// 17 MB row-pointer array is hit by every step and should stay -- without the hints ncu shows a 15 % L2 hit
// rate and three DRAM sectors per walk-step.
__device__ __forceinline__ uint64_t l2_policy_keep() {
    uint64_t pol;
    asm("createpolicy.fractional.L2::evict_last.b64 %0, 1.0;" : "=l"(pol));
    return pol;
}
__device__ __forceinline__ uint64_t l2_policy_stream() {
    uint64_t pol;
    asm("createpolicy.fractional.L2::evict_first.b64 %0, 1.0;" : "=l"(pol));
    return pol;
}
__device__ __forceinline__ int32_t ld_keep_s32(const int32_t *ptr, uint64_t pol) {
    int32_t v;  // not volatile: a read-only load the compiler may schedule freely among the other gathers
    asm("ld.global.nc.L2::cache_hint.s32 %0, [%1], %2;" : "=r"(v) : "l"(ptr), "l"(pol));
    return v;
}
__device__ __forceinline__ GrfEdge ld_stream_edge(const GrfEdge *ptr, uint64_t pol) {
    int4 raw;
    asm("ld.global.nc.L1::no_allocate.L2::cache_hint.v4.s32 {%0, %1, %2, %3}, [%4], %5;"
                 : "=r"(raw.x), "=r"(raw.y), "=r"(raw.z), "=r"(raw.w)
                 : "l"(ptr), "l"(pol));
    GrfEdge e;
    e.scaled = __hiloint2double(raw.y, raw.x);
    e.col = raw.z;
    e.pad = 0;
    return e;
}

template <bool kBlock>
__device__ __forceinline__ void group_sync() {
    if (kBlock)
        __syncthreads();
    else
        __syncwarp();
}

// exclusive scan of one int per thread over the group; `total` = group sum
template <bool kBlock>
__device__ __forceinline__ int group_excl_scan(int v, int *scratch, int &total) {
    const int lane = threadIdx.x & 31;
    int incl = v;
#pragma unroll
    for (int d = 1; d < 32; d <<= 1) {
        const int n = __shfl_up_sync(0xffffffffu, incl, d);
        if (lane >= d) incl += n;
    }
    if (!kBlock) {
        total = __shfl_sync(0xffffffffu, incl, 31);
        return incl - v;
    }
    const int warp = threadIdx.x >> 5;
    const int nwarps = blockDim.x >> 5;
    if (lane == 31) scratch[warp] = incl;
    __syncthreads();
    int before = 0, all = 0;
    for (int i = 0; i < nwarps; ++i) {
        const int s = scratch[i];
        if (i < warp) before += s;
        all += s;
    }
    __syncthreads();
    total = all;
    return before + incl - v;
}

// KPL = keys per lane of the warp-per-node variant (sort width 32*KPL >= W); 0 for the
// CTA-per-node variant, which sorts in shared memory.
#ifndef GRF_WALK_MINBLOCKS
#define GRF_WALK_MINBLOCKS 5  // register cap for the warp-per-node variant (walk-steps/s: grid config 2 | R-MAT 2^20 nodes)
// 1 or 4: 85 registers 97 G | 37 G;  5: 74 registers 102 G | 45 G;  6 or 7: 58-60 registers 102 G | 30 G
#endif
// kFast: Philox draws, cumulative load, per-edge factors precomputed (the production setting) --
// strips the per-step mode tests; the generic instantiation serves replay / ablation / sequential.
// kWide: a lane advances up to four of its walks together (graphs that miss L2: the walker is bound by DRAM
// latency and needs the independent gathers); otherwise one walk at a time (an L2-resident graph: the walker is
// bound by instruction issue, and the bookkeeping of four interleaved walks costs more than it hides).
// kStepSync (CTA-per-node only): the W walks of a start node advance one step at a time and every length is
// merged and written out before the next step, so shared memory holds ONE length's visit records (W x 12 bytes)
// instead of all L-1 of them -- the fallback for W x L beyond 227 KB (the reference's wind experiment runs
// W = 8192, L = 5, its ablation notebook W = 10000, L = 10).  Same draws, same arithmetic, same output.
template <bool kBlock, typename KeyT, int KPL, bool kFast, bool kWide, bool kStepSync>
__global__ void __launch_bounds__(kBlock ? 256 : 128, kBlock ? 1 : GRF_WALK_MINBLOCKS) walk_merge_kernel(const WalkParams p) {
    static_assert(!kStepSync || (kBlock && !kFast && !kWide), "step-synchronous walks: generic CTA variant only");
    constexpr int kIlp = !kWide ? 1 : (kBlock ? 4 : (KPL < 4 ? KPL : 4));
    const uint64_t keep = l2_policy_keep(), stream_pol = l2_policy_stream();
    extern __shared__ __align__(16) unsigned char smem_raw[];
    const int GS = kBlock ? (int)blockDim.x : 32;
    const int tg = kBlock ? (int)threadIdx.x : (int)(threadIdx.x & 31);
    const int groups_per_cta = kBlock ? 1 : (int)(blockDim.x >> 5);
    const int group_in_cta = kBlock ? 0 : (int)(threadIdx.x >> 5);

    unsigned char *base = smem_raw + (size_t)group_in_cta * p.group_bytes;
    double *loads = reinterpret_cast<double *>(base);                                  // [(L-1)][W]
    int32_t *nodes = reinterpret_cast<int32_t *>(base + p.loads_bytes);                // [(L-1)][W]
    double *sorted_loads = reinterpret_cast<double *>(base + p.loads_bytes + p.nodes_bytes);  // [32*KPL], warp variant
    KeyT *keys = reinterpret_cast<KeyT *>(base + p.loads_bytes + p.nodes_bytes + p.sorted_bytes);  // [Wp | 32*KPL]
    __shared__ int scan_scratch[32];

    const int W = p.W, L = p.L, Wp = p.Wp, wbits = p.wbits;
    const KeyT KEY_MAX = ~(KeyT)0;
    const KeyT wmask = ((KeyT)1 << wbits) - 1;
    const int chunk = (Wp + GS - 1) / GS;
    unsigned long long my_visits = 0;

    for (int64_t row = (int64_t)blockIdx.x * groups_per_cta + group_in_cta; row < p.n_local;
         row += (int64_t)gridDim.x * groups_per_cta) {
        const int64_t start = p.start_lo + row;

        // ---------------- phase 1: the walks -------------------------------
        if constexpr (kStepSync) {
            // the record of the current length doubles as the walker state: nodes[w] >= 0 = still walking
            for (int w = tg; w < W; w += GS) {
                nodes[w] = (int32_t)start;
                loads[w] = 1.0;
            }
            my_visits += (unsigned long long)((W - tg + GS - 1) / GS);  // the length-0 visits (start, 1.0)
        } else {
        // a walk that stops at length s leaves no visit at lengths > s: mark every slot empty first
        // (16-byte stores; per-walk tail loops cost 6 % of the kernel's instructions under ncu)
        {
            int4 *n4 = reinterpret_cast<int4 *>(nodes);
            const int n_vec = (int)(p.nodes_bytes >> 4);
            for (int i = tg; i < n_vec; i += GS) n4[i] = make_int4(-1, -1, -1, -1);
        }
        group_sync<kBlock>();
        // kIlp walks per lane advance in lockstep, one transition at a time: the row-pointer pairs of
        // all of them are requested first, then the edges -- kIlp independent gathers in flight per lane
        // instead of one dependent chain (config 4: the walker is bound by DRAM latency, ncu 9 warps
        // stalled on long scoreboard per issue with one walk per lane).
        for (int w0 = tg; w0 < W; w0 += GS * kIlp) {
            int32_t cur[kIlp];
            double load[kIlp];
            uint32_t x2[kIlp], x3[kIlp];  // second half of a Philox block, used by the odd step
            bool alive[kIlp];
#pragma unroll
            for (int r = 0; r < kIlp; ++r) {
                alive[r] = w0 + r * GS < W;
                cur[r] = (int32_t)start;
                load[r] = 1.0;
                x2[r] = x3[r] = 0u;
                my_visits += alive[r];  // the length-0 visit (start, 1.0)
            }
            for (int step = 0; step < L - 1; ++step) {
                int32_t rs[kIlp], deg[kIlp];
#pragma unroll
                for (int r = 0; r < kIlp; ++r) {
                    rs[r] = deg[r] = 0;
                    if (alive[r]) {
                        rs[r] = ld_keep_s32(p.row_ptr + cur[r], keep);
                        deg[r] = ld_keep_s32(p.row_ptr + cur[r] + 1, keep) - rs[r];
                    }
                }
                int64_t e[kIlp];
#pragma unroll
                for (int r = 0; r < kIlp; ++r) {
                    e[r] = 0;
                    if (!alive[r]) continue;
                    if (deg[r] == 0) {  // dead end: stop without drawing (sparse_sampler.py:47)
                        alive[r] = false;
                        continue;
                    }
                    const unsigned long long walk_id =
                        (unsigned long long)start * (unsigned long long)W + (unsigned)(w0 + r * GS);
                    int32_t k;
                    if (!kFast && p.draw_mode == GRF_DRAW_REPLAY) {
                        const long long ti = ((long long)walk_id - p.trace_base) * L + step;
                        if (__ldg(p.trace_u + ti) < p.p_halt) {
                            alive[r] = false;
                            continue;
                        }
                        k = __ldg(p.trace_k + ti);
                    } else {
                        // one Philox block serves two consecutive steps: words (0,1) the even one, (2,3) the odd one
                        uint32_t xh, xk;
                        if ((step & 1) == 0) {
                            uint32_t x[4];
                            philox4x32_10((uint32_t)walk_id, (uint32_t)(walk_id >> 32), (uint32_t)(step >> 1), 0u,
                                          p.k0, p.k1, x);
                            xh = x[0];
                            xk = x[1];
                            x2[r] = x[2];
                            x3[r] = x[3];
                        } else {
                            xh = x2[r];
                            xk = x3[r];
                        }
                        if ((unsigned long long)xh < p.halt_thr) {
                            alive[r] = false;
                            continue;
                        }
                        k = (int32_t)__umulhi(xk, (uint32_t)deg[r]);
                    }
                    e[r] = (int64_t)rs[r] + k;
                }
                // the edges: neighbour + load factor.  load *= degree * weight / (1 - p_halt), evaluated left
                // to right in float64 with no contraction (sparse_sampler.py:54); (deg * w) / (1 - p) depends
                // on the edge only, so grf_edge_records may have computed it once per edge (same roundings).
                int32_t nxt[kIlp];
                double fac[kIlp];
#pragma unroll
                for (int r = 0; r < kIlp; ++r) {
                    nxt[r] = 0;
                    fac[r] = 0.0;
                    if (!alive[r]) continue;
                    if (kFast || p.edges) {
                        const GrfEdge ed = ld_stream_edge(p.edges + e[r], stream_pol);
                        nxt[r] = ed.col;
                        fac[r] = ed.scaled;
                        if (!kFast && p.load_mode == GRF_LOAD_ABLATION) fac[r] = __ldg(p.val + e[r]);
                    } else {
                        nxt[r] = __ldg(p.col_idx + e[r]);
                        const double wv = __ldg(p.val + e[r]);
                        fac[r] = p.load_mode == GRF_LOAD_ABLATION
                                     ? wv
                                     : __ddiv_rn(__dmul_rn((double)deg[r], wv), p.one_minus_p);
                    }
                }
                bool any = false;
#pragma unroll
                for (int r = 0; r < kIlp; ++r) {
                    if (!alive[r]) continue;
                    load[r] = (kFast || p.load_mode == GRF_LOAD_CUMULATIVE) ? __dmul_rn(load[r], fac[r]) : fac[r];
                    cur[r] = nxt[r];
                    const int w = w0 + r * GS;
                    nodes[step * W + w] = cur[r];  // the visit at length step + 1
                    loads[step * W + w] = load[r];
                    ++my_visits;
                    any = true;
                }
                if (!any) break;
            }
        }
        }  // !kStepSync

        int32_t *out_col = p.stage_ent ? nullptr : p.stage_col + row * p.stride;
        double *out_sum = p.stage_ent ? nullptr : p.stage_sum + row * p.stride;
        GrfEntry *out_ent = p.stage_ent ? p.stage_ent + row * p.stride : nullptr;
        // one merged record: (column, unscaled float64 sum) for the reference layout, or the finished
        // float32 Phi entry -- (float)(sum * (1/W)) or (float)(sum / W), the arithmetic of grf_compact_blocks
        auto emit = [&](int slot, int32_t node, double sum, int length) {
            if (out_ent) {
                GrfEntry en;
                en.col = pack_col(node, length);
                en.val = (float)(p.scale_mode == GRF_SCALE_MUL_RECIP ? __dmul_rn(sum, p.recip_w)
                                                                      : __ddiv_rn(sum, p.w_as_double));
                out_ent[slot] = en;
            } else {
                out_col[slot] = node;
                out_sum[slot] = sum;
            }
        };
        if (tg == 0) {
            emit(0, (int32_t)start, (double)W, 0);  // M_0 = I: W visits of load 1.0, summed exactly
            p.row_cnt[row * L] = 1;
            if (p.col_counts) atomicAdd(p.col_counts + start * L, 1);
        }
        int off = 1;
        group_sync<kBlock>();

        // ---------------- phase 2: merge the visits of each length ----------
        for (int si = 0; si < L - 1; ++si) {
            const int rec = kStepSync ? 0 : si * W;  // where the visit records of length si + 1 live
            if constexpr (kStepSync) {
                // one transition of every walk that is still alive (the generic path of phase 1, one walk at a time)
                for (int w = tg; w < W; w += GS) {
                    const int32_t cur = nodes[w];
                    if (cur < 0) continue;
                    const int32_t rs = __ldg(p.row_ptr + cur);
                    const int32_t deg = __ldg(p.row_ptr + cur + 1) - rs;
                    if (deg == 0) {  // dead end: stop without drawing (sparse_sampler.py:47)
                        nodes[w] = -1;
                        continue;
                    }
                    const unsigned long long walk_id = (unsigned long long)start * (unsigned long long)W + (unsigned)w;
                    int32_t k;
                    if (p.draw_mode == GRF_DRAW_REPLAY) {
                        const long long ti = ((long long)walk_id - p.trace_base) * L + si;
                        if (__ldg(p.trace_u + ti) < p.p_halt) {
                            nodes[w] = -1;
                            continue;
                        }
                        k = __ldg(p.trace_k + ti);
                    } else {
                        uint32_t x[4];
                        philox4x32_10((uint32_t)walk_id, (uint32_t)(walk_id >> 32), (uint32_t)(si >> 1), 0u, p.k0,
                                      p.k1, x);
                        const uint32_t xh = (si & 1) ? x[2] : x[0], xk = (si & 1) ? x[3] : x[1];
                        if ((unsigned long long)xh < p.halt_thr) {
                            nodes[w] = -1;
                            continue;
                        }
                        k = (int32_t)__umulhi(xk, (uint32_t)deg);
                    }
                    const int64_t e = (int64_t)rs + k;
                    const double wv = __ldg(p.val + e);
                    const double fac = p.load_mode == GRF_LOAD_ABLATION
                                           ? wv
                                           : __ddiv_rn(__dmul_rn((double)deg, wv), p.one_minus_p);
                    nodes[w] = __ldg(p.col_idx + e);
                    loads[w] = p.load_mode == GRF_LOAD_CUMULATIVE ? __dmul_rn(loads[w], fac) : fac;
                    ++my_visits;
                }
                __syncthreads();
            }
            if constexpr (!kBlock) {
                // warp-per-node: sort in registers, park the sorted keys in shared memory
                // for the run walks below
                const int lane = tg;
                KeyT key[KPL];
#pragma unroll
                for (int r = 0; r < KPL; ++r) {
                    const int w = r * 32 + lane;
                    KeyT kk = KEY_MAX;
                    if (w < W) {
                        const int32_t nd = nodes[si * W + w];
                        if (nd >= 0) kk = ((KeyT)(uint32_t)nd << wbits) | (KeyT)w;
                    }
                    key[r] = kk;
                }
                // no walk reached this length (an isolated start node -- 42 % of the rows of the config-4 graph --
                // or every walk halted): none reaches a later one either.  Skips four 128-key sorts per such row
                // (ncu, config 4: the sort network was 22 % VIMNMX + 9 % SHFL of 22 warp-instructions per walk-step).
                {
                    bool have = false;
#pragma unroll
                    for (int r = 0; r < KPL; ++r) have |= key[r] != KEY_MAX;
                    if (!__any_sync(0xffffffffu, have)) {
                        if (lane == 0)
                            for (int s2 = si; s2 < L - 1; ++s2) p.row_cnt[row * L + s2 + 1] = 0;
                        break;
                    }
                }
                warp_bitonic_sort<KeyT, KPL>(key, lane);
                // park the loads in sorted order; a run (= one output entry) is then a contiguous
                // stretch of that stream.  Heads write their node and where their run starts; one lane
                // per run then adds the run's loads in walk order (the reference's summation order).
#pragma unroll
                for (int r = 0; r < KPL; ++r) {
                    const KeyT kk = key[r];
                    if (kk != KEY_MAX) sorted_loads[lane * KPL + r] = loads[si * W + (int)(kk & wmask)];
                }
                const KeyT prev_last = __shfl_up_sync(0xffffffffu, key[KPL - 1], 1);
                bool head[KPL];
                int counts = 0;  // heads in the low half, valid elements in the high half: one scan for both
#pragma unroll
                for (int r = 0; r < KPL; ++r) {
                    const KeyT kk = key[r];
                    const KeyT pv = r == 0 ? prev_last : key[r > 0 ? r - 1 : 0];
                    const bool first = (lane == 0 && r == 0);
                    head[r] = (kk != KEY_MAX) && (first || (pv >> wbits) != (kk >> wbits));
                    counts += (int)head[r] + ((int)(kk != KEY_MAX) << 16);
                }
                int totals;
                int rank = group_excl_scan<false>(counts, scan_scratch, totals) & 0xffff;
                const int total = totals & 0xffff, n_valid = totals >> 16;
                // run_start[j] = first sorted position of run j, run_node[j] = its node (the key area holds
                // 32 * KPL keys of >= 4 bytes: room for both int32 tables, runs <= 32 * KPL - 1 when n_valid
                // leaves one slot for the terminator; see the sizing of n_keys on the host)
                int32_t *run_start = reinterpret_cast<int32_t *>(keys);  // [total + 1]
                int32_t *run_node = run_start + 32 * KPL + 1;             // [total]
#pragma unroll
                for (int r = 0; r < KPL; ++r) {
                    if (head[r]) {
                        run_start[rank] = lane * KPL + r;
                        const int32_t node = (int32_t)(key[r] >> wbits);
                        run_node[rank] = node;
                        if (p.col_counts) atomicAdd(p.col_counts + (int64_t)node * L + si + 1, 1);
                        ++rank;
                    }
                }
                if (lane == 0) run_start[total] = n_valid;
                __syncwarp();
                for (int j = lane; j < total; j += 32) {
                    const int qb = run_start[j], qe = run_start[j + 1];
                    double sum = 0.0;
                    for (int q = qb; q < qe; ++q) sum = __dadd_rn(sum, sorted_loads[q]);
                    emit(off + j, run_node[j], sum, si + 1);
                }
                if (lane == 0) p.row_cnt[row * L + si + 1] = total;
                off += total;
                __syncwarp();
            } else {
                int have = 0;
                for (int i = tg; i < Wp; i += GS) {
                    KeyT key = KEY_MAX;
                    if (i < W) {
                        const int32_t nd = nodes[rec + i];
                        if (nd >= 0) key = ((KeyT)(uint32_t)nd << wbits) | (KeyT)i;
                    }
                    keys[i] = key;
                    have |= key != KEY_MAX;
                }
                if (!__syncthreads_or(have)) {  // nothing at this length, hence nothing at any later one
                    if (tg == 0)
                        for (int s2 = si; s2 < L - 1; ++s2) p.row_cnt[row * L + s2 + 1] = 0;
                    break;
                }
                for (uint32_t k = 2; k <= (uint32_t)Wp; k <<= 1) {
                    for (uint32_t j = k >> 1; j > 0; j >>= 1) {
                        for (uint32_t c = tg; c < (uint32_t)Wp / 2; c += GS) {
                            const uint32_t idx = ((c & ~(j - 1)) << 1) | (c & (j - 1));
                            const uint32_t ixj = idx | j;
                            const KeyT a = keys[idx], b = keys[ixj];
                            const bool up = (idx & k) == 0;
                            if ((a > b) == up) {
                                keys[idx] = b;
                                keys[ixj] = a;
                            }
                        }
                        __syncthreads();
                    }
                }
                // distinct nodes = run heads of the sorted keys; thread tg owns a
                // contiguous chunk so that ranks follow column order
                const int lo = tg * chunk;
                const int hi = min(Wp, lo + chunk);
                int heads = 0;
                for (int i = lo; i < hi; ++i) {
                    const KeyT key = keys[i];
                    if (key == KEY_MAX) break;
                    heads += (i == 0) || ((keys[i - 1] >> wbits) != (key >> wbits));
                }
                int total;
                int rank = group_excl_scan<true>(heads, scan_scratch, total);
                for (int i = lo; i < hi; ++i) {
                    const KeyT key = keys[i];
                    if (key == KEY_MAX) break;
                    const KeyT node = key >> wbits;
                    if ((i == 0) || ((keys[i - 1] >> wbits) != node)) {
                        double sum = 0.0;
                        for (int q = i; q < Wp; ++q) {
                            const KeyT kq = keys[q];
                            if ((kq >> wbits) != node) break;
                            sum = __dadd_rn(sum, loads[rec + (int)(kq & wmask)]);
                        }
                        emit(off + rank, (int32_t)node, sum, si + 1);
                        if (p.col_counts) atomicAdd(p.col_counts + (int64_t)node * L + si + 1, 1);
                        ++rank;
                    }
                }
                if (tg == 0) p.row_cnt[row * L + si + 1] = total;
                off += total;
                __syncthreads();
            }
        }
    }

    if (p.visits != nullptr) {
#pragma unroll
        for (int d = 16; d > 0; d >>= 1) my_visits += __shfl_xor_sync(0xffffffffu, my_visits, d);
        if ((threadIdx.x & 31) == 0 && my_visits) atomicAdd(p.visits, my_visits);
    }
}

template <bool kBlock, typename KeyT, int KPL, bool kFast = false, bool kWide = false, bool kStepSync = false>
static int launch_walk(const WalkParams &p, size_t smem, int threads, int grid, cudaStream_t stream) {
    auto kern = walk_merge_kernel<kBlock, KeyT, KPL, kFast, kWide, kStepSync>;
    GRF_CUDA_OK(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    kern<<<grid, threads, smem, stream>>>(p);
    return check_cuda(cudaGetLastError(), "walk_merge_kernel launch");
}

// ---------------- coupled walks (GRF_DRAW_COUPLE_HALT / GRF_DRAW_COUPLE_NEIGHBOURS) ----------------

// exclusive max of one int per thread over the preceding threads of the group (kReverse: the following
// ones); INT_MIN when there are none
template <bool kBlock, bool kReverse>
__device__ __forceinline__ int group_excl_max(int v, int *scratch) {
    const int lane = threadIdx.x & 31;
    int incl = v;
#pragma unroll
    for (int d = 1; d < 32; d <<= 1) {
        const int n = kReverse ? __shfl_down_sync(0xffffffffu, incl, d) : __shfl_up_sync(0xffffffffu, incl, d);
        if (kReverse ? lane + d < 32 : lane >= d) incl = max(incl, n);
    }
    int excl = kReverse ? __shfl_down_sync(0xffffffffu, incl, 1) : __shfl_up_sync(0xffffffffu, incl, 1);
    if (kReverse ? lane == 31 : lane == 0) excl = INT_MIN;
    if (!kBlock) return excl;
    const int warp = threadIdx.x >> 5;
    const int nwarps = blockDim.x >> 5;
    if (kReverse ? lane == 0 : lane == 31) scratch[warp] = incl;
    __syncthreads();
    for (int i = 0; i < nwarps; ++i)
        if (kReverse ? i > warp : i < warp) excl = max(excl, scratch[i]);
    __syncthreads();
    return excl;
}

// The W walks of a start node advance one step at a time (the kStepSync schedule of walk_merge_kernel, which
// this generalises).  Per length l: the visits are sorted by (node, walk) -- in registers when a warp owns the
// node (KPL keys per lane), in shared memory when a CTA does -- and parked as `keys`; every thread then owns
// the contiguous stretch [tg * chunk, tg * chunk + chunk) of the sorted order, and that one order serves
//   1. the merge: one entry per distinct node, loads added in walk order (the arithmetic of walk_merge_kernel);
//   2. the halting decisions of the walks at length l (partner's word for antithetic termination);
//   3. with repelling neighbours, a segmented rank / count of the continuing walks over the node runs:
//      j = continuing walks before this one at its node, m = continuing walks at its node, from one add scan
//      and two max scans (the cont-position of the last run head before and of the first run head after the
//      thread's stretch) -- no extra shared memory, so the W limit is the one-length limit of kStepSync;
//   4. the neighbour draws and edge gathers, which write the walker state of length l + 1.
// Between 2 and 4 nodes[w] is free (the keys hold the nodes) and carries (cont, head cont-position, j) of
// walk w; W < 2^15 (shared memory bounds it far below) keeps those in 15-bit fields.
template <bool kBlock, typename KeyT, int KPL>
__global__ void __launch_bounds__(kBlock ? 256 : 128) walk_coupled_kernel(const WalkParams p) {
    const uint64_t keep = l2_policy_keep(), stream_pol = l2_policy_stream();
    extern __shared__ __align__(16) unsigned char smem_raw[];
    const int GS = kBlock ? (int)blockDim.x : 32;
    const int tg = kBlock ? (int)threadIdx.x : (int)(threadIdx.x & 31);
    const int groups_per_cta = kBlock ? 1 : (int)(blockDim.x >> 5);
    const int group_in_cta = kBlock ? 0 : (int)(threadIdx.x >> 5);

    unsigned char *base = smem_raw + (size_t)group_in_cta * p.group_bytes;
    double *loads = reinterpret_cast<double *>(base);                                       // [W]
    int32_t *nodes = reinterpret_cast<int32_t *>(base + p.loads_bytes);                     // [W], -1 = stopped
    KeyT *keys = reinterpret_cast<KeyT *>(base + p.loads_bytes + p.nodes_bytes);            // [n_keys]
    __shared__ int scan_scratch[32];

    const int W = p.W, L = p.L, wbits = p.wbits;
    const int n_keys = kBlock ? p.Wp : 32 * KPL;
    const int chunk = n_keys / GS;
    const int lo = tg * chunk, hi = lo + chunk;
    const KeyT KEY_MAX = ~(KeyT)0;
    const KeyT wmask = ((KeyT)1 << wbits) - 1;
    const bool couple_halt = (p.draw_mode & GRF_DRAW_COUPLE_HALT) != 0;
    const bool repel = (p.draw_mode & GRF_DRAW_COUPLE_NEIGHBOURS) != 0;
    unsigned long long my_visits = 0;

    for (int64_t row = (int64_t)blockIdx.x * groups_per_cta + group_in_cta; row < p.n_local;
         row += (int64_t)gridDim.x * groups_per_cta) {
        const int64_t start = p.start_lo + row;
        for (int w = tg; w < W; w += GS) {
            nodes[w] = (int32_t)start;
            loads[w] = 1.0;
        }
        group_sync<kBlock>();

        int32_t *out_col = p.stage_ent ? nullptr : p.stage_col + row * p.stride;
        double *out_sum = p.stage_ent ? nullptr : p.stage_sum + row * p.stride;
        GrfEntry *out_ent = p.stage_ent ? p.stage_ent + row * p.stride : nullptr;
        auto emit = [&](int slot, int32_t node, double sum, int length) {
            if (out_ent) {
                GrfEntry en;
                en.col = pack_col(node, length);
                en.val = (float)(p.scale_mode == GRF_SCALE_MUL_RECIP ? __dmul_rn(sum, p.recip_w)
                                                                      : __ddiv_rn(sum, p.w_as_double));
                out_ent[slot] = en;
            } else {
                out_col[slot] = node;
                out_sum[slot] = sum;
            }
        };
        // walk w leaves node v (CSR row rs .. rs + deg) through neighbour index k: load update as
        // walk_merge_kernel's phase 1 (16-byte edge records when given)
        auto move = [&](int w, int32_t rs, int32_t deg, int32_t k) {
            const int64_t e = (int64_t)rs + k;
            int32_t nxt;
            double fac;
            if (p.edges) {
                const GrfEdge ed = ld_stream_edge(p.edges + e, stream_pol);
                nxt = ed.col;
                fac = p.load_mode == GRF_LOAD_ABLATION ? __ldg(p.val + e) : ed.scaled;
            } else {
                nxt = __ldg(p.col_idx + e);
                const double wv = __ldg(p.val + e);
                fac = p.load_mode == GRF_LOAD_ABLATION ? wv : __ddiv_rn(__dmul_rn((double)deg, wv), p.one_minus_p);
            }
            loads[w] = p.load_mode == GRF_LOAD_CUMULATIVE ? __dmul_rn(loads[w], fac) : fac;
            nodes[w] = nxt;
        };
        auto is_head = [&](int i, KeyT key) { return i == 0 || (keys[i - 1] >> wbits) != (key >> wbits); };

        int off = 0;
        for (int l = 0; l < L; ++l) {
            // ---- the visits of length l, sorted by (node, walk) ----
            if constexpr (!kBlock) {
                KeyT key[KPL];
                bool have = false;
#pragma unroll
                for (int r = 0; r < KPL; ++r) {
                    const int w = r * 32 + tg;
                    KeyT kk = KEY_MAX;
                    if (w < W) {
                        const int32_t nd = nodes[w];
                        if (nd >= 0) kk = ((KeyT)(uint32_t)nd << wbits) | (KeyT)w;
                    }
                    key[r] = kk;
                    have |= kk != KEY_MAX;
                }
                if (!__any_sync(0xffffffffu, have)) {  // every walk has stopped
                    if (tg == 0)
                        for (int s2 = l; s2 < L; ++s2) p.row_cnt[row * L + s2] = 0;
                    break;
                }
                warp_bitonic_sort<KeyT, KPL>(key, tg);
#pragma unroll
                for (int r = 0; r < KPL; ++r) keys[tg * KPL + r] = key[r];
                __syncwarp();
            } else {
                int have = 0;
                for (int i = tg; i < n_keys; i += GS) {
                    KeyT key = KEY_MAX;
                    if (i < W) {
                        const int32_t nd = nodes[i];
                        if (nd >= 0) key = ((KeyT)(uint32_t)nd << wbits) | (KeyT)i;
                    }
                    keys[i] = key;
                    have |= key != KEY_MAX;
                }
                if (!__syncthreads_or(have)) {
                    if (tg == 0)
                        for (int s2 = l; s2 < L; ++s2) p.row_cnt[row * L + s2] = 0;
                    break;
                }
                for (uint32_t k = 2; k <= (uint32_t)n_keys; k <<= 1) {
                    for (uint32_t j = k >> 1; j > 0; j >>= 1) {
                        for (uint32_t c = tg; c < (uint32_t)n_keys / 2; c += GS) {
                            const uint32_t idx = ((c & ~(j - 1)) << 1) | (c & (j - 1));
                            const uint32_t ixj = idx | j;
                            const KeyT a = keys[idx], b = keys[ixj];
                            const bool up = (idx & k) == 0;
                            if ((a > b) == up) {
                                keys[idx] = b;
                                keys[ixj] = a;
                            }
                        }
                        __syncthreads();
                    }
                }
            }

            // ---- 1. merge: one entry per distinct node, loads added in walk order ----
            int heads = 0;
            for (int i = lo; i < hi; ++i) {
                const KeyT key = keys[i];
                if (key == KEY_MAX) break;
                ++my_visits;
                heads += is_head(i, key);
            }
            int total;
            int rank = group_excl_scan<kBlock>(heads, scan_scratch, total);
            for (int i = lo; i < hi; ++i) {
                const KeyT key = keys[i];
                if (key == KEY_MAX) break;
                if (!is_head(i, key)) continue;
                const KeyT node = key >> wbits;
                double sum = 0.0;
                for (int q = i; q < n_keys; ++q) {
                    const KeyT kq = keys[q];
                    if ((kq >> wbits) != node) break;
                    sum = __dadd_rn(sum, loads[(int)(kq & wmask)]);
                }
                emit(off + rank, (int32_t)node, sum, l);
                if (p.col_counts) atomicAdd(p.col_counts + (int64_t)node * L + l, 1);
                ++rank;
            }
            if (tg == 0) p.row_cnt[row * L + l] = total;
            off += total;
            if (l == L - 1) break;
            group_sync<kBlock>();  // the merge has read every load: the moves below may overwrite them

            // ---- 2. halting decisions at step l ----
            int n_cont = 0, first_head = -1, last_head = -1;  // cont-positions (within the stretch) of run heads
            for (int i = lo; i < hi; ++i) {
                const KeyT key = keys[i];
                if (key == KEY_MAX) break;
                const int w = (int)(key & wmask);
                const int32_t v = (int32_t)(key >> wbits);
                if (is_head(i, key)) {
                    if (first_head < 0) first_head = n_cont;
                    last_head = n_cont;
                }
                const int32_t rs = ld_keep_s32(p.row_ptr + v, keep);
                const int32_t deg = ld_keep_s32(p.row_ptr + v + 1, keep) - rs;
                bool cont = false;
                if (deg > 0) {  // a dead end stops the walk without a draw
                    const int src = (couple_halt && (w & 1)) ? w - 1 : w;  // walk 2q+1 halts on walk 2q's word
                    const unsigned long long gid = (unsigned long long)start * (unsigned long long)W + (unsigned)src;
                    uint32_t x[4];
                    philox4x32_10((uint32_t)gid, (uint32_t)(gid >> 32), (uint32_t)(l >> 1), 0u, p.k0, p.k1, x);
                    const uint32_t xh = ((l & 1) ? x[2] : x[0]) ^ (src != w ? 0x80000000u : 0u);
                    cont = (unsigned long long)xh >= p.halt_thr;
                    if (cont && !repel) {  // independent neighbour: the walk's own word
                        if (src != w) {
                            const unsigned long long own = gid + 1;
                            philox4x32_10((uint32_t)own, (uint32_t)(own >> 32), (uint32_t)(l >> 1), 0u, p.k0, p.k1,
                                          x);
                        }
                        const uint32_t xk = (l & 1) ? x[3] : x[1];
                        move(w, rs, deg, (int32_t)__umulhi(xk, (uint32_t)deg));
                    }
                }
                if (repel)
                    nodes[w] = cont;
                else if (!cont)
                    nodes[w] = -1;
                n_cont += cont;
            }
            if (repel) {
                // ---- 3. segmented rank / count of the continuing walks over the node runs ----
                int n_all;
                const int cpos0 = group_excl_scan<kBlock>(n_cont, scan_scratch, n_all);
                const int head_before = group_excl_max<kBlock, false>(last_head >= 0 ? cpos0 + last_head : INT_MIN,
                                                                      scan_scratch);
                const int neg_head_after = group_excl_max<kBlock, true>(
                    first_head >= 0 ? -(cpos0 + first_head) : INT_MIN, scan_scratch);
                // forward: cont-position hc of the walk's run head and j = its own cont-position - hc
                int c = cpos0, hc = head_before;
                for (int i = lo; i < hi; ++i) {
                    const KeyT key = keys[i];
                    if (key == KEY_MAX) break;
                    const int w = (int)(key & wmask);
                    if (is_head(i, key)) hc = c;
                    const int cont = nodes[w];
                    nodes[w] = (cont << 30) | (hc << 15) | (c - hc);
                    c += cont;
                }
                // backward: ec = cont-position of the next run head (or the total), m = ec - hc; the moves
                int ec = neg_head_after == INT_MIN ? n_all : -neg_head_after;
                for (int i = hi - 1; i >= lo; --i) {
                    const KeyT key = keys[i];
                    if (key == KEY_MAX) continue;
                    const int w = (int)(key & wmask);
                    const int32_t v = (int32_t)(key >> wbits);
                    const int packed = nodes[w];
                    const int hcw = (packed >> 15) & 0x7fff, j = packed & 0x7fff;
                    if (packed >> 30) {
                        const int m = ec - hcw;
                        const int32_t rs = ld_keep_s32(p.row_ptr + v, keep);
                        const int32_t deg = ld_keep_s32(p.row_ptr + v + 1, keep) - rs;
                        uint32_t x[4];
                        philox4x32_10((uint32_t)start, (uint32_t)v, (uint32_t)l, 1u, p.k0, p.k1, x);
                        const uint64_t cg = __umulhi(x[0], (uint32_t)deg);
                        const uint64_t k = (cg + (uint64_t)j * (uint64_t)deg / (uint64_t)m) % (uint64_t)deg;
                        move(w, rs, deg, (int32_t)k);
                    } else {
                        nodes[w] = -1;
                    }
                    if (is_head(i, key)) ec = hcw;
                }
            }
            group_sync<kBlock>();  // the state of length l + 1 is complete
        }
        group_sync<kBlock>();  // every read of this row's keys and loads is done before the next row
    }

    if (p.visits != nullptr) {
#pragma unroll
        for (int d = 16; d > 0; d >>= 1) my_visits += __shfl_xor_sync(0xffffffffu, my_visits, d);
        if ((threadIdx.x & 31) == 0 && my_visits) atomicAdd(p.visits, my_visits);
    }
}

template <bool kBlock, typename KeyT, int KPL>
static int launch_coupled(const WalkParams &p, size_t smem, int threads, int grid, cudaStream_t stream) {
    auto kern = walk_coupled_kernel<kBlock, KeyT, KPL>;
    GRF_CUDA_OK(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    kern<<<grid, threads, smem, stream>>>(p);
    return check_cuda(cudaGetLastError(), "walk_coupled_kernel launch");
}

// The coupled draws take the step-synchronous schedule: shared memory holds one length's visit records
// (W x 12 bytes) and the sort keys.  W <= 256: a warp per start node, four per CTA; else a CTA per start node.
static int walk_coupled(WalkParams &p, bool key32, int64_t n_nodes, cudaStream_t st) {
    const size_t key_size = key32 ? 4 : 8;
    const size_t kMaxSmem = 227 * 1024 - 256;
    p.loads_bytes = (uint32_t)(((size_t)p.W * 8 + 15) & ~(size_t)15);
    p.nodes_bytes = (uint32_t)(((size_t)p.W * 4 + 15) & ~(size_t)15);
    p.sorted_bytes = 0;
    if (p.W <= 256) {
        const int kpl = p.Wp <= 32 ? 1 : p.Wp / 32;
        const size_t gb = ((size_t)p.loads_bytes + p.nodes_bytes + (size_t)32 * kpl * key_size + 15) & ~(size_t)15;
        p.group_bytes = (uint32_t)gb;
        const int warps = 4;
        const int64_t want = (p.n_local + warps - 1) / warps;
        const int grid = (int)(want < (int64_t)kSmCount * 64 ? want : (int64_t)kSmCount * 64);
        const size_t smem = warps * gb;
        const int threads = warps * 32;
#define GRF_COUPLED_CASE(K)                                                                  \
    case K:                                                                                  \
        return key32 ? launch_coupled<false, uint32_t, K>(p, smem, threads, grid, st)       \
                     : launch_coupled<false, unsigned long long, K>(p, smem, threads, grid, st)
        switch (kpl) {
            GRF_COUPLED_CASE(1);
            GRF_COUPLED_CASE(2);
            GRF_COUPLED_CASE(4);
            default:
                GRF_COUPLED_CASE(8);
        }
#undef GRF_COUPLED_CASE
    }
    const size_t gb = ((size_t)p.loads_bytes + p.nodes_bytes + (size_t)p.Wp * key_size + 15) & ~(size_t)15;
    if (gb > kMaxSmem)
        return fail(GRF_ERR_UNSUPPORTED,
                    "grf_walk: W=%d needs %zu B of shared memory per start node for one walk length (max %zu; "
                    "%d-byte sort keys for %lld nodes)", p.W, gb, kMaxSmem, (int)key_size, (long long)n_nodes);
    p.group_bytes = (uint32_t)gb;
    const int grid = (int)(p.n_local < (int64_t)kSmCount * 32 ? p.n_local : (int64_t)kSmCount * 32);
    return key32 ? launch_coupled<true, uint32_t, 0>(p, gb, 256, grid, st)
                 : launch_coupled<true, unsigned long long, 0>(p, gb, 256, grid, st);
}

}  // namespace grf

extern "C" int64_t grf_walk_stage_stride(int32_t walks_per_node, int32_t max_walk_length) {
    if (walks_per_node < 1 || max_walk_length < 1) return 0;
    return 1 + (int64_t)(max_walk_length - 1) * (int64_t)walks_per_node;
}

extern "C" int grf_walk(const GrfGraph *graph, const GrfWalkCfg *cfg, int64_t stage_stride, int32_t *stage_col,
                        double *stage_sum, int32_t *row_cnt, unsigned long long *visits_out, void *stream) {
    GRF_ON_STREAM_DEVICE(stream, row_cnt);
    using namespace grf;
    GRF_REQUIRE(graph && cfg, "grf_walk: null graph/cfg");
    GRF_REQUIRE(graph->n_nodes >= 0 && graph->n_nodes < (1ll << 31), "grf_walk: n_nodes %lld out of int32 range",
                (long long)graph->n_nodes);
    GRF_REQUIRE(graph->nnz >= 0 && graph->nnz < (1ll << 31), "grf_walk: nnz %lld out of int32 range",
                (long long)graph->nnz);
    GRF_REQUIRE(cfg->walks_per_node >= 1, "grf_walk: walks_per_node must be >= 1");
    GRF_REQUIRE(cfg->max_walk_length >= 1, "grf_walk: max_walk_length must be >= 1");
    GRF_REQUIRE(cfg->p_halt >= 0.0 && cfg->p_halt <= 1.0, "grf_walk: p_halt must be in [0, 1]");
    GRF_REQUIRE(cfg->start_lo >= 0 && cfg->start_lo <= cfg->start_hi && cfg->start_hi <= graph->n_nodes,
                "grf_walk: start range [%lld, %lld) outside [0, %lld)", (long long)cfg->start_lo,
                (long long)cfg->start_hi, (long long)graph->n_nodes);
    const int32_t coupled = GRF_DRAW_COUPLE_HALT | GRF_DRAW_COUPLE_NEIGHBOURS;
    GRF_REQUIRE((cfg->draw_mode & ~(GRF_DRAW_REPLAY | coupled)) == 0, "grf_walk: bad draw_mode");
    GRF_REQUIRE(!(cfg->draw_mode & GRF_DRAW_REPLAY) || !(cfg->draw_mode & coupled),
                "grf_walk: coupled draws need native Philox draws");
    GRF_REQUIRE(cfg->load_mode >= GRF_LOAD_CUMULATIVE && cfg->load_mode <= GRF_LOAD_ABLATION,
                "grf_walk: bad load_mode");
    GRF_REQUIRE(cfg->draw_mode != GRF_DRAW_REPLAY || (cfg->trace_u && cfg->trace_k),
                "grf_walk: replay mode needs trace_u and trace_k");
    GRF_REQUIRE(stage_stride >= grf_walk_stage_stride(cfg->walks_per_node, cfg->max_walk_length),
                "grf_walk: stage_stride too small");
    const int64_t n_local = cfg->start_hi - cfg->start_lo;
    if (n_local == 0) return GRF_OK;
    GRF_REQUIRE(graph->row_ptr && row_cnt && (cfg->stage_entries || (stage_col && stage_sum)), "grf_walk: null buffer");
    GRF_REQUIRE(cfg->scale_mode == GRF_SCALE_MUL_RECIP || cfg->scale_mode == GRF_SCALE_DIV, "grf_walk: bad scale_mode");
    GRF_REQUIRE(graph->nnz == 0 || (graph->col_idx && graph->val), "grf_walk: null edge arrays");

    WalkParams p;
    p.row_ptr = graph->row_ptr;
    p.col_idx = graph->col_idx;
    p.val = graph->val;
    p.edges = cfg->edges;
    p.trace_base = cfg->trace_walk_base;
    p.stage_ent = cfg->stage_entries;
    p.scale_mode = cfg->scale_mode;
    p.recip_w = 1.0 / (double)cfg->walks_per_node;
    p.w_as_double = (double)cfg->walks_per_node;
    p.start_lo = cfg->start_lo;
    p.n_local = n_local;
    p.W = cfg->walks_per_node;
    p.L = cfg->max_walk_length;
    p.Wp = (int32_t)next_pow2((uint32_t)p.W);
    p.wbits = bit_width((uint64_t)p.Wp - 1);
    p.p_halt = cfg->p_halt;
    p.one_minus_p = 1.0 - cfg->p_halt;
    double thr = floor(cfg->p_halt * 4294967296.0);
    thr = thr < 0.0 ? 0.0 : (thr > 4294967296.0 ? 4294967296.0 : thr);
    p.halt_thr = (unsigned long long)thr;
    p.k0 = (uint32_t)cfg->seed;
    p.k1 = (uint32_t)(cfg->seed >> 32);
    p.draw_mode = cfg->draw_mode;
    p.load_mode = cfg->load_mode;
    p.trace_u = cfg->trace_u;
    p.trace_k = cfg->trace_k;
    p.stride = stage_stride;
    p.stage_col = stage_col;
    p.stage_sum = stage_sum;
    p.row_cnt = row_cnt;
    p.visits = visits_out;
    p.col_counts = cfg->col_counts;

    const int node_bits = bit_width((uint64_t)(graph->n_nodes > 0 ? graph->n_nodes - 1 : 0));
    const bool key32 = node_bits + p.wbits <= 31;
    const size_t key_size = key32 ? 4 : 8;
    const size_t steps = (size_t)(p.L - 1);
    p.loads_bytes = (uint32_t)((steps * p.W * 8 + 15) & ~(size_t)15);  // keeps `nodes` 16-byte aligned
    p.nodes_bytes = (uint32_t)((steps * p.W * 4 + 15) & ~(size_t)15);  // whole int4s: the kernel clears it with 16-byte stores
    const bool warp_variant = p.W <= 256;
    const int kpl = p.Wp <= 32 ? 1 : p.Wp / 32;  // warp variant sorts 32*kpl keys
    const size_t n_keys = warp_variant ? (size_t)32 * kpl : (size_t)p.Wp;
    p.sorted_bytes = warp_variant ? (uint32_t)(n_keys * 8) : 0u;
    // the warp variant sorts in registers and reuses the key area as run_start[n_keys + 1] + run_node[n_keys]
    const size_t key_area = warp_variant ? (2 * n_keys + 1) * 4 : n_keys * key_size;
    const size_t gb = ((size_t)p.loads_bytes + p.nodes_bytes + p.sorted_bytes + key_area + 15) & ~(size_t)15;
    p.group_bytes = (uint32_t)gb;
    const size_t kMaxSmem = 227 * 1024 - 256;
    GRF_REQUIRE((uint64_t)p.W * (uint64_t)p.L < (1ull << 31), "grf_walk: W*L too large");

    cudaStream_t st = (cudaStream_t)stream;
    if (cfg->draw_mode & coupled) return walk_coupled(p, key32, graph->n_nodes, st);
    // start nodes per CTA of the warp-per-node variant: as many of 4, 2, 1 as the visit records leave room for
    // (W = 200, L = 30: one group is 68 KB); none fits -> the CTA-per-node variants below
    int warps = 4;
    while (warps > 1 && warps * gb > kMaxSmem) warps >>= 1;
    if (warp_variant && warps * gb <= kMaxSmem) {
        const int64_t want = (n_local + warps - 1) / warps;
        const int grid = (int)(want < (int64_t)kSmCount * 64 ? want : (int64_t)kSmCount * 64);
        const size_t smem = warps * gb;
        const int threads = warps * 32;
        const bool fast = p.draw_mode == GRF_DRAW_PHILOX && p.load_mode == GRF_LOAD_CUMULATIVE && p.edges;
        // the edge records of this graph do not fit L2 (126 MB, shared with staging writes): latency-bound regime
        const char *ilp_env = getenv("GRF_B200_WALK_WIDE");
        const bool wide = ilp_env ? ilp_env[0] == '1' : graph->nnz * (int64_t)sizeof(GrfEdge) > (48ll << 20);
#define GRF_WALK_CASE(K)                                                                                    \
    case K:                                                                                                 \
        if (fast && wide)                                                                                   \
            return key32 ? launch_walk<false, uint32_t, K, true, true>(p, smem, threads, grid, st)         \
                         : launch_walk<false, unsigned long long, K, true, true>(p, smem, threads, grid, st); \
        if (fast)                                                                                           \
            return key32 ? launch_walk<false, uint32_t, K, true>(p, smem, threads, grid, st)               \
                         : launch_walk<false, unsigned long long, K, true>(p, smem, threads, grid, st);     \
        return key32 ? launch_walk<false, uint32_t, K>(p, smem, threads, grid, st)                         \
                     : launch_walk<false, unsigned long long, K>(p, smem, threads, grid, st)
        switch (kpl) {
            GRF_WALK_CASE(1);
            GRF_WALK_CASE(2);
            GRF_WALK_CASE(4);
            default:
                GRF_WALK_CASE(8);
        }
#undef GRF_WALK_CASE
    }
    const int64_t want = n_local;
    const int grid = (int)(want < (int64_t)kSmCount * 32 ? want : (int64_t)kSmCount * 32);
    // CTA per start node, shared-memory sort of Wp keys (the warp variant's layout does not apply)
    const size_t cta_keys = (size_t)p.Wp * key_size;
    const size_t gb_cta = ((size_t)p.loads_bytes + p.nodes_bytes + cta_keys + 15) & ~(size_t)15;
    if (gb_cta <= kMaxSmem) {
        p.sorted_bytes = 0;
        p.group_bytes = (uint32_t)gb_cta;
        return key32 ? launch_walk<true, uint32_t, 0, false, true>(p, gb_cta, 256, grid, st)
                     : launch_walk<true, unsigned long long, 0, false, true>(p, gb_cta, 256, grid, st);
    }
    // all lengths do not fit: one length at a time (W x 12 bytes of records + the sort keys)
    p.loads_bytes = (uint32_t)(((size_t)p.W * 8 + 15) & ~(size_t)15);
    p.nodes_bytes = (uint32_t)(((size_t)p.W * 4 + 15) & ~(size_t)15);
    p.sorted_bytes = 0;
    const size_t gb_ss = ((size_t)p.loads_bytes + p.nodes_bytes + cta_keys + 15) & ~(size_t)15;
    if (gb_ss > kMaxSmem)
        return fail(GRF_ERR_UNSUPPORTED,
                    "grf_walk: W=%d needs %zu B of shared memory per start node for one walk length (max %zu; "
                    "%d-byte sort keys for %lld nodes)", p.W, gb_ss, kMaxSmem, (int)key_size,
                    (long long)graph->n_nodes);
    p.group_bytes = (uint32_t)gb_ss;
    return key32 ? launch_walk<true, uint32_t, 0, false, false, true>(p, gb_ss, 256, grid, st)
                 : launch_walk<true, unsigned long long, 0, false, false, true>(p, gb_ss, 256, grid, st);
}

namespace grf {
__global__ void __launch_bounds__(256) edge_records_kernel(const int32_t *__restrict__ row_ptr,
                                                           const int32_t *__restrict__ col,
                                                           const double *__restrict__ val, int64_t n_nodes,
                                                           double one_minus_p, GrfEdge *__restrict__ out) {
    const int lane = threadIdx.x & 31;
    const int64_t warp0 = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    const int64_t nwarps = ((int64_t)gridDim.x * blockDim.x) >> 5;
    for (int64_t r = warp0; r < n_nodes; r += nwarps) {
        const int32_t b = row_ptr[r], e = row_ptr[r + 1];
        const double deg = (double)(e - b);
        // eight batches of a row in flight (a hub row of 175 303 neighbours is 5 500 batches for one warp)
        constexpr int kU = 8;
        for (int32_t i0 = b + lane; i0 < e; i0 += 32 * kU) {
            double v[kU];
            int32_t c[kU];
#pragma unroll
            for (int u = 0; u < kU; ++u) {
                const int32_t i = i0 + 32 * u;
                v[u] = i < e ? val[i] : 0.0;
                c[u] = i < e ? col[i] : 0;
            }
#pragma unroll
            for (int u = 0; u < kU; ++u) {
                const int32_t i = i0 + 32 * u;
                if (i >= e) continue;
                GrfEdge ed;
                ed.scaled = __ddiv_rn(__dmul_rn(deg, v[u]), one_minus_p);
                ed.col = c[u];
                ed.pad = 0;
                out[i] = ed;
            }
        }
    }
}
}  // namespace grf

extern "C" int grf_edge_records(const GrfGraph *graph, double p_halt, GrfEdge *edges, void *stream) {
    GRF_ON_STREAM_DEVICE(stream, edges);
    using namespace grf;
    GRF_REQUIRE(graph, "grf_edge_records: null graph");
    GRF_REQUIRE(p_halt >= 0.0 && p_halt <= 1.0, "grf_edge_records: p_halt must be in [0, 1]");
    if (graph->n_nodes == 0 || graph->nnz == 0) return GRF_OK;
    GRF_REQUIRE(graph->row_ptr && graph->col_idx && graph->val && edges, "grf_edge_records: null buffer");
    int64_t g = (graph->n_nodes + 7) / 8;
    if (g > (int64_t)kSmCount * 32) g = (int64_t)kSmCount * 32;
    edge_records_kernel<<<(int)g, 256, 0, (cudaStream_t)stream>>>(graph->row_ptr, graph->col_idx, graph->val,
                                                                 graph->n_nodes, 1.0 - p_halt, edges);
    return check_cuda(cudaGetLastError(), "edge_records_kernel launch");
}
