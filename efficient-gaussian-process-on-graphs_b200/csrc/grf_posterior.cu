// Exact GP posterior variance on the GRF features (no reference counterpart: the reference's users estimate the
// variance from SparseGraphGP.predict samples).  With the training rows Phi_f[x] touching the column set S, the
// whitened training features C = G L^-T (G = Phi_f[x]^T restricted to S, L L^T = G^T G + sigma^2 I) live on S,
// and the variance at a test node needs one pass over its row of Phi_f:
//     q_i = sum_{c < r} ( sum_{e in row x*_i, slot(col e) >= 0} w_e C[slot(col e), c] )^2,   d_i = sum_e w_e^2,
// w_e = f[length(e)] * e.val.  The factor itself is a handful of float64 cuBLAS / cuSOLVER calls
// (grf_b200/posterior.py); the pass over every candidate row is this file.
//
// One warp per test row, grid-stride.  The warp streams the row's entries once: d in float64, the slot lookup,
// and the touched entries compacted as (slot, w) pairs into a per-warp shared buffer (ballot + prefix, so in row
// order).  Then, per panel of 128 columns of C, every lane holds a float4 of column sums, gathers the C rows of the
// listed slots (16-byte loads when C and ldc allow it), and at the end of the panel squares and adds its sums into a
// float64.  A row with more touched entries than the buffer holds re-streams its entries per panel, one buffer at
// a time, in the same order.  Every sum has a fixed order and there are no atomics, so repeated calls agree bit for
// bit.

#include "grf_common.cuh"

namespace grf {
namespace {

constexpr int kQfWarps = 8;        // warps per CTA
constexpr int kQfCap = 256;        // (slot, w) pairs per warp buffer
constexpr int kQfPanel = 128;      // columns of C per panel: a float4 per lane

struct QfPair {
    int32_t slot;
    float w;
};

// s += sum over the listed pairs of w * C[slot, c .. c + 3] (only columns < r are read when the loads are scalar; a
// 16-byte load may read columns [r, round_up(r, 4)) of a row, whose sums never reach a result)
template <bool VEC>
__device__ __forceinline__ void qf_gather(const QfPair *buf, int cnt, const float *__restrict__ C, int64_t ldc,
                                          int32_t c, int32_t r, float4 &s) {
    if (c >= r) return;
    if (VEC) {
        int j = 0;
        for (; j + 4 <= cnt; j += 4) {
            float4 v[4];
            float w[4];
#pragma unroll
            for (int u = 0; u < 4; ++u) {
                const QfPair p = buf[j + u];
                w[u] = p.w;
                v[u] = __ldg(reinterpret_cast<const float4 *>(C + (int64_t)p.slot * ldc + c));
            }
#pragma unroll
            for (int u = 0; u < 4; ++u) {
                s.x = fmaf(w[u], v[u].x, s.x);
                s.y = fmaf(w[u], v[u].y, s.y);
                s.z = fmaf(w[u], v[u].z, s.z);
                s.w = fmaf(w[u], v[u].w, s.w);
            }
        }
        for (; j < cnt; ++j) {
            const QfPair p = buf[j];
            const float4 v = __ldg(reinterpret_cast<const float4 *>(C + (int64_t)p.slot * ldc + c));
            s.x = fmaf(p.w, v.x, s.x);
            s.y = fmaf(p.w, v.y, s.y);
            s.z = fmaf(p.w, v.z, s.z);
            s.w = fmaf(p.w, v.w, s.w);
        }
    } else {
        // columns past r - 1 load column r - 1 again: in bounds, and qf_square drops those sums
        const int o1 = min(1, r - 1 - c), o2 = min(2, r - 1 - c), o3 = min(3, r - 1 - c);
        for (int j = 0; j < cnt; ++j) {
            const QfPair p = buf[j];
            const float *row = C + (int64_t)p.slot * ldc + c;
            s.x = fmaf(p.w, __ldg(row), s.x);
            s.y = fmaf(p.w, __ldg(row + o1), s.y);
            s.z = fmaf(p.w, __ldg(row + o2), s.z);
            s.w = fmaf(p.w, __ldg(row + o3), s.w);
        }
    }
}

// sum of the squares of the sums of columns < r, in float64
__device__ __forceinline__ double qf_square(const float4 &s, int32_t c, int32_t r) {
    double acc = 0.0;
    if (c < r) acc += (double)s.x * (double)s.x;
    if (c + 1 < r) acc += (double)s.y * (double)s.y;
    if (c + 2 < r) acc += (double)s.z * (double)s.z;
    if (c + 3 < r) acc += (double)s.w * (double)s.w;
    return acc;
}

// Compacts the touched entries of ent[k0, k0 + 32) ∩ [k0, end) into buf[cnt ..), in row order; returns the number
// of touched entries of the group (they are stored only below kQfCap).  With D, also adds w^2 of every entry to d.
template <bool D>
__device__ __forceinline__ int qf_compact(const int2 *__restrict__ ent2, int32_t k0, int32_t end,
                                          const float *fs, const int32_t *__restrict__ col_slot, QfPair *buf, int cnt,
                                          int lane, double &d) {
    const int32_t k = k0 + lane;
    int32_t slot = -1;
    float w = 0.f;
    if (k < end) {
        const int2 e = __ldg(ent2 + k);
        w = fs[entry_step(e.x)] * __int_as_float(e.y);
        slot = __ldg(col_slot + entry_col(e.x));
        if (D) d += (double)w * (double)w;
    }
    const unsigned hit = __ballot_sync(0xffffffffu, slot >= 0);
    const int pos = cnt + __popc(hit & ((1u << lane) - 1u));
    if (slot >= 0 && pos < kQfCap) buf[pos] = QfPair{slot, w};
    return __popc(hit);
}

template <bool VEC>
__global__ void __launch_bounds__(kQfWarps * 32) row_quadform_kernel(
    const int32_t *__restrict__ ptr, const GrfEntry *__restrict__ ent, const float *__restrict__ f, int32_t L,
    const int32_t *__restrict__ x, int64_t n, int64_t row_lo, int64_t n_rows, const int32_t *__restrict__ col_slot,
    const float *__restrict__ C, int64_t ldc, int32_t r, float *__restrict__ q, float *__restrict__ d_out) {
    __shared__ float fs[kMaxSteps];
    __shared__ QfPair sbuf[kQfWarps][kQfCap];
    if (threadIdx.x < kMaxSteps) fs[threadIdx.x] = threadIdx.x < L ? __ldg(f + threadIdx.x) : 0.f;
    __syncthreads();
    const int lane = threadIdx.x & 31;
    QfPair *buf = sbuf[threadIdx.x >> 5];
    const int64_t warp0 = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    const int64_t n_warps = ((int64_t)gridDim.x * blockDim.x) >> 5;
    const int2 *ent2 = reinterpret_cast<const int2 *>(ent);
    for (int64_t i = warp0; i < n; i += n_warps) {
        const int64_t a = (x ? (int64_t)__ldg(x + i) : i + row_lo) - row_lo;
        double dsum = 0.0, qsum = 0.0;
        if (a >= 0 && a < n_rows) {   // rows outside this shard stay +0
            const int32_t b = __ldg(ptr + a * L), e = __ldg(ptr + (a + 1) * L);
            // one pass: d, and the touched entries into the buffer (the first kQfCap of them)
            int cnt = 0;
            for (int32_t k0 = b; k0 < e; k0 += 32)
                cnt += qf_compact<true>(ent2, k0, e, fs, col_slot, buf, cnt, lane, dsum);
            __syncwarp();
            if (cnt <= kQfCap) {
                for (int32_t c0 = 0; c0 < r; c0 += kQfPanel) {
                    const int32_t c = c0 + 4 * lane;
                    float4 s = make_float4(0.f, 0.f, 0.f, 0.f);
                    qf_gather<VEC>(buf, cnt, C, ldc, c, r, s);
                    qsum += qf_square(s, c, r);
                }
            } else {
                // long row: per panel, re-stream the entries one buffer at a time (same order as above)
                for (int32_t c0 = 0; c0 < r; c0 += kQfPanel) {
                    const int32_t c = c0 + 4 * lane;
                    float4 s = make_float4(0.f, 0.f, 0.f, 0.f);
                    int part = 0;
                    for (int32_t k0 = b; k0 < e; k0 += 32) {
                        if (part + 32 > kQfCap) {
                            __syncwarp();
                            qf_gather<VEC>(buf, part, C, ldc, c, r, s);
                            __syncwarp();
                            part = 0;
                        }
                        part += qf_compact<false>(ent2, k0, e, fs, col_slot, buf, part, lane, dsum);
                    }
                    __syncwarp();
                    qf_gather<VEC>(buf, part, C, ldc, c, r, s);
                    __syncwarp();
                    qsum += qf_square(s, c, r);
                }
            }
            __syncwarp();   // the buffer is reused by the next row
#pragma unroll
            for (int o = 16; o > 0; o >>= 1) {
                dsum += __shfl_xor_sync(0xffffffffu, dsum, o);
                qsum += __shfl_xor_sync(0xffffffffu, qsum, o);
            }
        }
        if (lane == 0) {
            q[i] = (float)qsum;
            if (d_out) d_out[i] = (float)dsum;
        }
    }
}

// ---- row projection: out[i, c] = sum_{e in row x[i], slot >= 0} w_e B[slot(e), c] -------------------------------
// The posterior mean (r = 1), samples (r up to 64) and covariance (r = n) are this product.  Three warp shapes,
// chosen by r (profiles/prof_row_project_shapes.py compares them with a build that takes the panels for every r):
//   r <= 4   row_project_narrow_kernel: lanes own entries.  In the panel form one lane of 32 would gather B for
//            every touched entry of the row in a serial chain of dependent loads (power-law hub rows hold 10^4 and
//            more); here every lane gathers its own entries, four rounds of loads in flight at a time.
//   <= 64    row_project_mid_kernel: entry groups x column quads, so the gather chain of a row is split over the
//            groups instead of running in the few lanes whose columns are < r.
//   r > 64   row_project_kernel: the panels of row_quadform_kernel (128 columns, a float4 of column sums per
//            lane), stored instead of squared (16-byte stores when out and ldo allow it); long rows re-stream per
//            panel in the same order.
// Each fixes its summation order and uses no atomics, so repeated calls agree bit for bit.

// columns [c, min(c + 4, r)) of s into the output row o
__device__ __forceinline__ void pj_store(float *__restrict__ o, int32_t c, int32_t r, const float4 &s, bool vec) {
    if (c >= r) return;
    if (vec && c + 4 <= r) {
        *reinterpret_cast<float4 *>(o + c) = s;
        return;
    }
    o[c] = s.x;
    if (c + 1 < r) o[c + 1] = s.y;
    if (c + 2 < r) o[c + 2] = s.z;
    if (c + 3 < r) o[c + 3] = s.w;
}

// r <= 4: lane l adds w * B[slot, 0 .. 3] for its entries l, l + 32, l + 64, ... in that order, with the loads of
// kNarrowRounds rounds issued before their sums; the warp then adds the lanes with a fixed xor tree (every lane ends
// with the same bits) and lane c stores column c.  With VEC a 16-byte load reads B[slot, 0 .. 3] (ldb % 4 == 0, so
// those columns lie inside the row); otherwise columns past r - 1 load column r - 1 again, and are never stored.
constexpr int kNarrowRounds = 4;

// the lane's share of the narrow sums over the entries [b, e) of one row (o1 .. o3 as in the kernel)
template <bool VEC>
__device__ __forceinline__ void pj_narrow_row(const int2 *__restrict__ ent2, int32_t b, int32_t e, const float *fs,
                                              const int32_t *__restrict__ col_slot, const float *__restrict__ B,
                                              int64_t ldb, int lane, int o1, int o2, int o3, float4 &s) {
    for (int32_t k0 = b + lane; k0 < e; k0 += 32 * kNarrowRounds) {
        int2 en[kNarrowRounds];
        int32_t slot[kNarrowRounds];
        float4 v[kNarrowRounds];
#pragma unroll
        for (int u = 0; u < kNarrowRounds; ++u)
            en[u] = k0 + 32 * u < e ? __ldg(ent2 + k0 + 32 * u) : make_int2(0, 0);
#pragma unroll
        for (int u = 0; u < kNarrowRounds; ++u)
            slot[u] = k0 + 32 * u < e ? __ldg(col_slot + entry_col(en[u].x)) : -1;
#pragma unroll
        for (int u = 0; u < kNarrowRounds; ++u) {
            v[u] = make_float4(0.f, 0.f, 0.f, 0.f);
            if (slot[u] >= 0) {
                const float *row = B + (int64_t)slot[u] * ldb;
                if (VEC) {
                    v[u] = __ldg(reinterpret_cast<const float4 *>(row));
                } else {
                    v[u].x = __ldg(row);
                    v[u].y = __ldg(row + o1);
                    v[u].z = __ldg(row + o2);
                    v[u].w = __ldg(row + o3);
                }
            }
        }
#pragma unroll
        for (int u = 0; u < kNarrowRounds; ++u) {
            if (slot[u] >= 0) {
                const float w = fs[entry_step(en[u].x)] * __int_as_float(en[u].y);
                s.x = fmaf(w, v[u].x, s.x);
                s.y = fmaf(w, v[u].y, s.y);
                s.z = fmaf(w, v[u].z, s.z);
                s.w = fmaf(w, v[u].w, s.w);
            }
        }
    }
}

template <bool VEC>
__global__ void __launch_bounds__(kQfWarps * 32) row_project_narrow_kernel(
    const int32_t *__restrict__ ptr, const GrfEntry *__restrict__ ent, const float *__restrict__ f, int32_t L,
    const int32_t *__restrict__ x, int64_t n, int64_t row_lo, int64_t n_rows, const int32_t *__restrict__ col_slot,
    const float *__restrict__ B, int64_t ldb, int32_t r, float *__restrict__ out, int64_t ldo) {
    __shared__ float fs[kMaxSteps];
    if (threadIdx.x < kMaxSteps) fs[threadIdx.x] = threadIdx.x < L ? __ldg(f + threadIdx.x) : 0.f;
    __syncthreads();
    const int lane = threadIdx.x & 31;
    const int64_t warp0 = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    const int64_t n_warps = ((int64_t)gridDim.x * blockDim.x) >> 5;
    const int2 *ent2 = reinterpret_cast<const int2 *>(ent);
    const int o1 = min(1, r - 1), o2 = min(2, r - 1), o3 = min(3, r - 1);
    for (int64_t i = warp0; i < n; i += n_warps) {
        const int64_t a = (x ? (int64_t)__ldg(x + i) : i + row_lo) - row_lo;
        float4 s = make_float4(0.f, 0.f, 0.f, 0.f);
        if (a >= 0 && a < n_rows) {   // rows outside this shard stay +0
            const int32_t b = __ldg(ptr + a * L), e = __ldg(ptr + (a + 1) * L);
            pj_narrow_row<VEC>(ent2, b, e, fs, col_slot, B, ldb, lane, o1, o2, o3, s);
        }
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) {
            s.x += __shfl_xor_sync(0xffffffffu, s.x, o);
            s.y += __shfl_xor_sync(0xffffffffu, s.y, o);
            s.z += __shfl_xor_sync(0xffffffffu, s.z, o);
            s.w += __shfl_xor_sync(0xffffffffu, s.w, o);
        }
        if (lane < r) out[i * ldo + lane] = lane == 0 ? s.x : lane == 1 ? s.y : lane == 2 ? s.z : s.w;
    }
}

// s += w * B[slot, c .. c + 3]: a 16-byte load, or scalar loads of columns < r (columns past r - 1 load column
// r - 1 again, whose sums pj_store drops)
template <bool VEC>
__device__ __forceinline__ void pj_fma(const float *__restrict__ B, int64_t ldb, int32_t slot, float w, int32_t c,
                                       int32_t r, float4 &s) {
    const float *row = B + (int64_t)slot * ldb + c;
    if (VEC) {
        const float4 v = __ldg(reinterpret_cast<const float4 *>(row));
        s.x = fmaf(w, v.x, s.x);
        s.y = fmaf(w, v.y, s.y);
        s.z = fmaf(w, v.z, s.z);
        s.w = fmaf(w, v.w, s.w);
    } else {
        const int o1 = min(1, r - 1 - c), o2 = min(2, r - 1 - c), o3 = min(3, r - 1 - c);
        s.x = fmaf(w, __ldg(row), s.x);
        s.y = fmaf(w, __ldg(row + o1), s.y);
        s.z = fmaf(w, __ldg(row + o2), s.z);
        s.w = fmaf(w, __ldg(row + o3), s.w);
    }
}

// 4 < r <= 64: group g of the 32 / Q entry groups adds the buffered pairs g, g + 32 / Q, ... (Q column quads,
// Q = 1 << qlog); four pairs' loads in flight at a time
template <bool VEC>
__device__ __forceinline__ void pj_gather_groups(const QfPair *buf, int cnt, int grp, int step,
                                                 const float *__restrict__ B, int64_t ldb, int32_t c, int32_t r,
                                                 float4 &s) {
    if (c >= r) return;
    int j = grp;
    for (; j + 3 * step < cnt; j += 4 * step) {
        QfPair p[4];
#pragma unroll
        for (int u = 0; u < 4; ++u) p[u] = buf[j + u * step];
#pragma unroll
        for (int u = 0; u < 4; ++u) pj_fma<VEC>(B, ldb, p[u].slot, p[u].w, c, r, s);
    }
    for (; j < cnt; j += step) {
        const QfPair p = buf[j];
        pj_fma<VEC>(B, ldb, p.slot, p.w, c, r, s);
    }
}

// the group's share of the mid sums over the entries [b, e) of one row: compaction, then the gathers (re-streamed
// in buffer loads when the row has more touched entries than the buffer)
template <bool VEC>
__device__ __forceinline__ void pj_mid_row(const int2 *__restrict__ ent2, int32_t b, int32_t e, const float *fs,
                                           const int32_t *__restrict__ col_slot, QfPair *buf, int grp, int step,
                                           const float *__restrict__ B, int64_t ldb, int32_t c, int32_t r, int lane,
                                           double &unused, float4 &s) {
    int cnt = 0;
    for (int32_t k0 = b; k0 < e; k0 += 32)
        cnt += qf_compact<false>(ent2, k0, e, fs, col_slot, buf, cnt, lane, unused);
    __syncwarp();
    if (cnt <= kQfCap) {
        pj_gather_groups<VEC>(buf, cnt, grp, step, B, ldb, c, r, s);
    } else {
        int part = 0;
        for (int32_t k0 = b; k0 < e; k0 += 32) {
            if (part + 32 > kQfCap) {
                __syncwarp();
                pj_gather_groups<VEC>(buf, part, grp, step, B, ldb, c, r, s);
                __syncwarp();
                part = 0;
            }
            part += qf_compact<false>(ent2, k0, e, fs, col_slot, buf, part, lane, unused);
        }
        __syncwarp();
        pj_gather_groups<VEC>(buf, part, grp, step, B, ldb, c, r, s);
    }
    __syncwarp();   // the buffer is reused by the next row
}

// 4 < r <= 64: the warp is 32 / Q entry groups x Q column quads (Q the next power of two >= r / 4).  The touched
// pairs are compacted as in row_quadform_kernel, each group gathers its share, the groups are added with a fixed
// xor tree and group 0 stores.  Rows with more touched entries than the buffer re-stream in buffer loads.
template <bool VEC>
__global__ void __launch_bounds__(kQfWarps * 32) row_project_mid_kernel(
    const int32_t *__restrict__ ptr, const GrfEntry *__restrict__ ent, const float *__restrict__ f, int32_t L,
    const int32_t *__restrict__ x, int64_t n, int64_t row_lo, int64_t n_rows, const int32_t *__restrict__ col_slot,
    const float *__restrict__ B, int64_t ldb, int32_t r, float *__restrict__ out, int64_t ldo, int32_t qlog,
    bool vec_out) {
    __shared__ float fs[kMaxSteps];
    __shared__ QfPair sbuf[kQfWarps][kQfCap];
    if (threadIdx.x < kMaxSteps) fs[threadIdx.x] = threadIdx.x < L ? __ldg(f + threadIdx.x) : 0.f;
    __syncthreads();
    const int lane = threadIdx.x & 31;
    const int grp = lane >> qlog, step = 32 >> qlog;
    const int32_t c = 4 * (lane & ((1 << qlog) - 1));
    QfPair *buf = sbuf[threadIdx.x >> 5];
    const int64_t warp0 = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    const int64_t n_warps = ((int64_t)gridDim.x * blockDim.x) >> 5;
    const int2 *ent2 = reinterpret_cast<const int2 *>(ent);
    double unused = 0.0;
    for (int64_t i = warp0; i < n; i += n_warps) {
        const int64_t a = (x ? (int64_t)__ldg(x + i) : i + row_lo) - row_lo;
        float4 s = make_float4(0.f, 0.f, 0.f, 0.f);
        if (a >= 0 && a < n_rows) {   // rows outside this shard stay +0
            const int32_t b = __ldg(ptr + a * L), e = __ldg(ptr + (a + 1) * L);
            pj_mid_row<VEC>(ent2, b, e, fs, col_slot, buf, grp, step, B, ldb, c, r, lane, unused, s);
        }
        for (int o = 16; o >= (1 << qlog); o >>= 1) {
            s.x += __shfl_xor_sync(0xffffffffu, s.x, o);
            s.y += __shfl_xor_sync(0xffffffffu, s.y, o);
            s.z += __shfl_xor_sync(0xffffffffu, s.z, o);
            s.w += __shfl_xor_sync(0xffffffffu, s.w, o);
        }
        if (grp == 0) pj_store(out + i * ldo, c, r, s, vec_out);
    }
}

template <bool VEC>
__global__ void __launch_bounds__(kQfWarps * 32) row_project_kernel(
    const int32_t *__restrict__ ptr, const GrfEntry *__restrict__ ent, const float *__restrict__ f, int32_t L,
    const int32_t *__restrict__ x, int64_t n, int64_t row_lo, int64_t n_rows, const int32_t *__restrict__ col_slot,
    const float *__restrict__ B, int64_t ldb, int32_t r, float *__restrict__ out, int64_t ldo, bool vec_out) {
    __shared__ float fs[kMaxSteps];
    __shared__ QfPair sbuf[kQfWarps][kQfCap];
    if (threadIdx.x < kMaxSteps) fs[threadIdx.x] = threadIdx.x < L ? __ldg(f + threadIdx.x) : 0.f;
    __syncthreads();
    const int lane = threadIdx.x & 31;
    QfPair *buf = sbuf[threadIdx.x >> 5];
    const int64_t warp0 = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    const int64_t n_warps = ((int64_t)gridDim.x * blockDim.x) >> 5;
    const int2 *ent2 = reinterpret_cast<const int2 *>(ent);
    double unused = 0.0;
    for (int64_t i = warp0; i < n; i += n_warps) {
        const int64_t a = (x ? (int64_t)__ldg(x + i) : i + row_lo) - row_lo;
        int32_t b = 0, e = 0;                 // rows outside this shard: no entries, a row of +0
        if (a >= 0 && a < n_rows) {
            b = __ldg(ptr + a * L);
            e = __ldg(ptr + (a + 1) * L);
        }
        int cnt = 0;
        for (int32_t k0 = b; k0 < e; k0 += 32)
            cnt += qf_compact<false>(ent2, k0, e, fs, col_slot, buf, cnt, lane, unused);
        __syncwarp();
        float *o = out + i * ldo;
        for (int32_t c0 = 0; c0 < r; c0 += kQfPanel) {
            const int32_t c = c0 + 4 * lane;
            float4 s = make_float4(0.f, 0.f, 0.f, 0.f);
            if (cnt <= kQfCap) {
                qf_gather<VEC>(buf, cnt, B, ldb, c, r, s);
            } else {
                int part = 0;
                for (int32_t k0 = b; k0 < e; k0 += 32) {
                    if (part + 32 > kQfCap) {
                        __syncwarp();
                        qf_gather<VEC>(buf, part, B, ldb, c, r, s);
                        __syncwarp();
                        part = 0;
                    }
                    part += qf_compact<false>(ent2, k0, e, fs, col_slot, buf, part, lane, unused);
                }
                __syncwarp();
                qf_gather<VEC>(buf, part, B, ldb, c, r, s);
                __syncwarp();
            }
            pj_store(o, c, r, s, vec_out);
        }
        __syncwarp();   // the buffer is reused by the next row
    }
}

// ---- rank-k conditioning of the variance (and mean) at fixed candidate rows ---------------------------------------
// After the posterior gains b training rows, C gains b columns and a changes (grf_b200/posterior.py, condition_on);
// the variance at a candidate only drops by the squares of its projection onto the new columns.  With k = r +
// with_mean columns of B = [C_new | a]:
//     p_c(i) = sum_{e in row x[i], slot >= 0} w_e B[slot(e), c],   q[i] += sum_{c < r} p_c(i)^2   (float64, c = 0, 1, ..),
//     var[i] = max((float)(d[i] - q[i]), +0) (NaN stays NaN),       mean[i] = p_r(i).
// The sums p are those of the projection shapes (narrow for k <= 4, mid for k <= 64), in the same order; lane 0
// then adds the squares to q in column order, so repeated calls agree bit for bit.  Ids outside the shard have
// p = 0: q is left as it is, var is still written.

// lane 0: q += s_c^2 (DOWN: q -= s_c^2) for the columns c .. c + 3 below r, and the mean from column r when it is
// one of them
template <bool DOWN>
__device__ __forceinline__ void rc_add(double &qv, float &mv, const float4 &s, int32_t c, int32_t r) {
    const float v[4] = {s.x, s.y, s.z, s.w};
#pragma unroll
    for (int u = 0; u < 4; ++u) {
        if (c + u < r) {
            if (DOWN) qv -= (double)v[u] * (double)v[u];
            else qv += (double)v[u] * (double)v[u];
        } else if (c + u == r) {
            mv = v[u];
        }
    }
}

__device__ __forceinline__ float rc_var(float d, double q) {
    const float v = (float)((double)d - q);
    return v > 0.f || v != v ? v : 0.f;   // clamped at +0; NaN propagates as in torch.clamp_min
}

template <bool VEC, bool DOWN>
__device__ __forceinline__ void rc_narrow(
    const int32_t *__restrict__ ptr, const GrfEntry *__restrict__ ent, const float *__restrict__ f, int32_t L,
    const int32_t *__restrict__ x, int64_t n, int64_t row_lo, int64_t n_rows, const int32_t *__restrict__ col_slot,
    const float *__restrict__ B, int64_t ldb, int32_t k, int32_t r, double *__restrict__ q,
    const float *__restrict__ d, float *__restrict__ var, float *__restrict__ mean) {
    __shared__ float fs[kMaxSteps];
    if (threadIdx.x < kMaxSteps) fs[threadIdx.x] = threadIdx.x < L ? __ldg(f + threadIdx.x) : 0.f;
    __syncthreads();
    const int lane = threadIdx.x & 31;
    const int64_t warp0 = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    const int64_t n_warps = ((int64_t)gridDim.x * blockDim.x) >> 5;
    const int2 *ent2 = reinterpret_cast<const int2 *>(ent);
    const int o1 = min(1, k - 1), o2 = min(2, k - 1), o3 = min(3, k - 1);
    for (int64_t i = warp0; i < n; i += n_warps) {
        const int64_t a = (x ? (int64_t)__ldg(x + i) : i + row_lo) - row_lo;
        const bool inside = a >= 0 && a < n_rows;
        float4 s = make_float4(0.f, 0.f, 0.f, 0.f);
        if (inside) {
            const int32_t b = __ldg(ptr + a * L), e = __ldg(ptr + (a + 1) * L);
            pj_narrow_row<VEC>(ent2, b, e, fs, col_slot, B, ldb, lane, o1, o2, o3, s);
        }
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) {
            s.x += __shfl_xor_sync(0xffffffffu, s.x, o);
            s.y += __shfl_xor_sync(0xffffffffu, s.y, o);
            s.z += __shfl_xor_sync(0xffffffffu, s.z, o);
            s.w += __shfl_xor_sync(0xffffffffu, s.w, o);
        }
        if (lane == 0) {
            double qv = q[i];
            float mv = 0.f;
            if (inside) {
                rc_add<DOWN>(qv, mv, s, 0, r);
                q[i] = qv;
            }
            var[i] = rc_var(__ldg(d + i), qv);
            if (mean) mean[i] = mv;
        }
    }
}

// 4 < k <= 64: the groups x quads of row_project_mid_kernel; after the group tree, lane 0 collects the quads of
// group 0 in column order
template <bool VEC, bool DOWN>
__device__ __forceinline__ void rc_mid(
    const int32_t *__restrict__ ptr, const GrfEntry *__restrict__ ent, const float *__restrict__ f, int32_t L,
    const int32_t *__restrict__ x, int64_t n, int64_t row_lo, int64_t n_rows, const int32_t *__restrict__ col_slot,
    const float *__restrict__ B, int64_t ldb, int32_t k, int32_t r, double *__restrict__ q,
    const float *__restrict__ d, float *__restrict__ var, float *__restrict__ mean, int32_t qlog) {
    __shared__ float fs[kMaxSteps];
    __shared__ QfPair sbuf[kQfWarps][kQfCap];
    if (threadIdx.x < kMaxSteps) fs[threadIdx.x] = threadIdx.x < L ? __ldg(f + threadIdx.x) : 0.f;
    __syncthreads();
    const int lane = threadIdx.x & 31;
    const int grp = lane >> qlog, step = 32 >> qlog;
    const int32_t c = 4 * (lane & ((1 << qlog) - 1));
    const int nq = (k + 3) / 4;
    QfPair *buf = sbuf[threadIdx.x >> 5];
    const int64_t warp0 = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    const int64_t n_warps = ((int64_t)gridDim.x * blockDim.x) >> 5;
    const int2 *ent2 = reinterpret_cast<const int2 *>(ent);
    double unused = 0.0;
    for (int64_t i = warp0; i < n; i += n_warps) {
        const int64_t a = (x ? (int64_t)__ldg(x + i) : i + row_lo) - row_lo;
        const bool inside = a >= 0 && a < n_rows;
        float4 s = make_float4(0.f, 0.f, 0.f, 0.f);
        if (inside) {
            const int32_t b = __ldg(ptr + a * L), e = __ldg(ptr + (a + 1) * L);
            pj_mid_row<VEC>(ent2, b, e, fs, col_slot, buf, grp, step, B, ldb, c, k, lane, unused, s);
        }
        for (int o = 16; o >= (1 << qlog); o >>= 1) {
            s.x += __shfl_xor_sync(0xffffffffu, s.x, o);
            s.y += __shfl_xor_sync(0xffffffffu, s.y, o);
            s.z += __shfl_xor_sync(0xffffffffu, s.z, o);
            s.w += __shfl_xor_sync(0xffffffffu, s.w, o);
        }
        double qv = lane == 0 ? q[i] : 0.0;
        float mv = 0.f;
#pragma unroll 1
        for (int j = 0; j < nq; ++j) {   // quad j of group 0 sits in lane j
            float4 t;
            t.x = __shfl_sync(0xffffffffu, s.x, j);
            t.y = __shfl_sync(0xffffffffu, s.y, j);
            t.z = __shfl_sync(0xffffffffu, s.z, j);
            t.w = __shfl_sync(0xffffffffu, s.w, j);
            if (inside) rc_add<DOWN>(qv, mv, t, 4 * j, r);
        }
        if (lane == 0) {
            if (inside) q[i] = qv;
            var[i] = rc_var(__ldg(d + i), qv);
            if (mean) mean[i] = mv;
        }
    }
}

// The kernels: DOWN = false adds the squares (grf_phi_row_condition), DOWN = true subtracts them
// (grf_phi_row_downdate).  Same bodies, so a downdate sums p in exactly the order of the condition pass.
#define GRF_RC_ARGS                                                                                          \
    const int32_t *__restrict__ ptr, const GrfEntry *__restrict__ ent, const float *__restrict__ f, int32_t L,     \
        const int32_t *__restrict__ x, int64_t n, int64_t row_lo, int64_t n_rows,                                  \
        const int32_t *__restrict__ col_slot, const float *__restrict__ B, int64_t ldb, int32_t k, int32_t r,      \
        double *__restrict__ q, const float *__restrict__ d, float *__restrict__ var, float *__restrict__ mean
#define GRF_RC_PASS ptr, ent, f, L, x, n, row_lo, n_rows, col_slot, B, ldb, k, r, q, d, var, mean

template <bool VEC>
__global__ void __launch_bounds__(kQfWarps * 32) row_condition_narrow_kernel(GRF_RC_ARGS) {
    rc_narrow<VEC, false>(GRF_RC_PASS);
}

template <bool VEC>
__global__ void __launch_bounds__(kQfWarps * 32) row_downdate_narrow_kernel(GRF_RC_ARGS) {
    rc_narrow<VEC, true>(GRF_RC_PASS);
}

template <bool VEC>
__global__ void __launch_bounds__(kQfWarps * 32) row_condition_mid_kernel(GRF_RC_ARGS, int32_t qlog) {
    rc_mid<VEC, false>(GRF_RC_PASS, qlog);
}

template <bool VEC>
__global__ void __launch_bounds__(kQfWarps * 32) row_downdate_mid_kernel(GRF_RC_ARGS, int32_t qlog) {
    rc_mid<VEC, true>(GRF_RC_PASS, qlog);
}

#undef GRF_RC_PASS
#undef GRF_RC_ARGS

}  // namespace
}  // namespace grf

using namespace grf;

extern "C" int grf_phi_row_quadform(const GrfPhi *phi, const float *f, const int32_t *x, int64_t n,
                                    const int32_t *col_slot, const float *C, int64_t ldc, int32_t r, float *q,
                                    float *d, void *stream) {
    GRF_ON_STREAM_DEVICE(stream, q);
    GRF_REQUIRE(phi && f && col_slot && C && q, "grf_phi_row_quadform: null argument");
    GRF_REQUIRE(n >= 0 && r >= 0 && ldc >= r, "grf_phi_row_quadform: bad n / r / ldc");
    GRF_REQUIRE(phi->n_steps >= 1 && phi->n_steps <= kMaxSteps, "grf_phi_row_quadform: n_steps out of range");
    GRF_REQUIRE(x || n == phi->n_rows, "grf_phi_row_quadform: n must equal n_rows when x is NULL");
    if (n == 0) return GRF_OK;
    GRF_REQUIRE(phi->blk_ptr, "grf_phi_row_quadform: Phi blocks missing");
    const bool vec = ldc % 4 == 0 && ((uintptr_t)C & 15u) == 0;
    int64_t g = (n + kQfWarps - 1) / kQfWarps;
    if (g > (int64_t)kSmCount * 16) g = (int64_t)kSmCount * 16;
    cudaStream_t st = (cudaStream_t)stream;
    if (vec)
        row_quadform_kernel<true><<<(int)g, kQfWarps * 32, 0, st>>>(phi->blk_ptr, phi->entries, f, phi->n_steps, x,
                                                                    n, phi->row_lo, phi->n_rows, col_slot, C, ldc, r,
                                                                    q, d);
    else
        row_quadform_kernel<false><<<(int)g, kQfWarps * 32, 0, st>>>(phi->blk_ptr, phi->entries, f, phi->n_steps,
                                                                     x, n, phi->row_lo, phi->n_rows, col_slot, C,
                                                                     ldc, r, q, d);
    return check_cuda(cudaGetLastError(), "row_quadform_kernel launch");
}

extern "C" int grf_phi_row_project(const GrfPhi *phi, const float *f, const int32_t *x, int64_t n,
                                   const int32_t *col_slot, const float *B, int64_t ldb, int32_t r, float *out,
                                   int64_t ldo, void *stream) {
    GRF_ON_STREAM_DEVICE(stream, out);
    GRF_REQUIRE(phi && f && col_slot && B && out, "grf_phi_row_project: null argument");
    GRF_REQUIRE(n >= 0 && r >= 0 && ldb >= r && ldo >= r, "grf_phi_row_project: bad n / r / ldb / ldo");
    GRF_REQUIRE(phi->n_steps >= 1 && phi->n_steps <= kMaxSteps, "grf_phi_row_project: n_steps out of range");
    GRF_REQUIRE(x || n == phi->n_rows, "grf_phi_row_project: n must equal n_rows when x is NULL");
    GRF_REQUIRE(phi->blk_ptr, "grf_phi_row_project: Phi blocks missing");
    if (n == 0 || r == 0) return GRF_OK;
    const bool vin = ldb % 4 == 0 && ((uintptr_t)B & 15u) == 0;
    const bool vout = ldo % 4 == 0 && ((uintptr_t)out & 15u) == 0;
    int64_t g = (n + kQfWarps - 1) / kQfWarps;
    if (g > (int64_t)kSmCount * 16) g = (int64_t)kSmCount * 16;
    const dim3 grid((unsigned)g), block(kQfWarps * 32);
    cudaStream_t st = (cudaStream_t)stream;
    const int32_t *ptr = phi->blk_ptr;
    const GrfEntry *ent = phi->entries;
    const int32_t L = phi->n_steps;
    if (r <= 4) {
        if (vin)
            row_project_narrow_kernel<true><<<grid, block, 0, st>>>(ptr, ent, f, L, x, n, phi->row_lo, phi->n_rows,
                                                                    col_slot, B, ldb, r, out, ldo);
        else
            row_project_narrow_kernel<false><<<grid, block, 0, st>>>(ptr, ent, f, L, x, n, phi->row_lo, phi->n_rows,
                                                                     col_slot, B, ldb, r, out, ldo);
        return check_cuda(cudaGetLastError(), "row_project_narrow_kernel launch");
    }
    if (r <= 64) {
        int qlog = 1;                         // quads: the next power of two >= ceil(r / 4), 2 .. 16
        while ((4 << qlog) < r) ++qlog;
        if (vin)
            row_project_mid_kernel<true><<<grid, block, 0, st>>>(ptr, ent, f, L, x, n, phi->row_lo, phi->n_rows,
                                                                 col_slot, B, ldb, r, out, ldo, qlog, vout);
        else
            row_project_mid_kernel<false><<<grid, block, 0, st>>>(ptr, ent, f, L, x, n, phi->row_lo, phi->n_rows,
                                                                  col_slot, B, ldb, r, out, ldo, qlog, vout);
        return check_cuda(cudaGetLastError(), "row_project_mid_kernel launch");
    }
    if (vin)
        row_project_kernel<true><<<grid, block, 0, st>>>(ptr, ent, f, L, x, n, phi->row_lo, phi->n_rows, col_slot, B,
                                                         ldb, r, out, ldo, vout);
    else
        row_project_kernel<false><<<grid, block, 0, st>>>(ptr, ent, f, L, x, n, phi->row_lo, phi->n_rows, col_slot, B,
                                                          ldb, r, out, ldo, vout);
    return check_cuda(cudaGetLastError(), "row_project_kernel launch");
}

// grf_phi_row_condition (DOWN = false) and grf_phi_row_downdate (DOWN = true): the same arguments and rules
template <bool DOWN>
static int row_update(const char *name, const GrfPhi *phi, const float *f, const int32_t *x, int64_t n,
                      const int32_t *col_slot, const float *B, int64_t ldb, int32_t r, int32_t with_mean, double *q,
                      const float *d, float *var, float *mean, void *stream) {
    GRF_ON_STREAM_DEVICE(stream, var);
    GRF_REQUIRE(phi && f && col_slot && B && q && d && var && (mean || !with_mean), "%s: null argument", name);
    GRF_REQUIRE(with_mean == 0 || with_mean == 1, "%s: with_mean must be 0 or 1", name);
    const int64_t k = (int64_t)r + with_mean;
    GRF_REQUIRE(n >= 0 && r >= 0 && k >= 1 && k <= 64 && ldb >= k,
                "%s: bad n / r / ldb (needs 1 <= r + with_mean <= 64 and ldb >= r + with_mean)", name);
    GRF_REQUIRE(phi->n_steps >= 1 && phi->n_steps <= kMaxSteps, "%s: n_steps out of range", name);
    GRF_REQUIRE(x || n == phi->n_rows, "%s: n must equal n_rows when x is NULL", name);
    GRF_REQUIRE(phi->blk_ptr, "%s: Phi blocks missing", name);
    if (n == 0) return GRF_OK;
    const bool vin = ldb % 4 == 0 && ((uintptr_t)B & 15u) == 0;
    int64_t g = (n + kQfWarps - 1) / kQfWarps;
    if (g > (int64_t)kSmCount * 16) g = (int64_t)kSmCount * 16;
    const dim3 grid((unsigned)g), block(kQfWarps * 32);
    cudaStream_t st = (cudaStream_t)stream;
    const int32_t *ptr = phi->blk_ptr;
    const GrfEntry *ent = phi->entries;
    const int32_t L = phi->n_steps, kk = (int32_t)k;
    float *mo = with_mean ? mean : nullptr;
    if (k <= 4) {
        auto kern = DOWN ? (vin ? row_downdate_narrow_kernel<true> : row_downdate_narrow_kernel<false>)
                         : (vin ? row_condition_narrow_kernel<true> : row_condition_narrow_kernel<false>);
        kern<<<grid, block, 0, st>>>(ptr, ent, f, L, x, n, phi->row_lo, phi->n_rows, col_slot, B, ldb, kk, r, q, d,
                                     var, mo);
        return check_cuda(cudaGetLastError(),
                          DOWN ? "row_downdate_narrow_kernel launch" : "row_condition_narrow_kernel launch");
    }
    int qlog = 1;                             // quads: the next power of two >= ceil(k / 4), 2 .. 16
    while ((4 << qlog) < k) ++qlog;
    auto kern = DOWN ? (vin ? row_downdate_mid_kernel<true> : row_downdate_mid_kernel<false>)
                     : (vin ? row_condition_mid_kernel<true> : row_condition_mid_kernel<false>);
    kern<<<grid, block, 0, st>>>(ptr, ent, f, L, x, n, phi->row_lo, phi->n_rows, col_slot, B, ldb, kk, r, q, d, var,
                                 mo, qlog);
    return check_cuda(cudaGetLastError(), DOWN ? "row_downdate_mid_kernel launch" : "row_condition_mid_kernel launch");
}

extern "C" int grf_phi_row_condition(const GrfPhi *phi, const float *f, const int32_t *x, int64_t n,
                                     const int32_t *col_slot, const float *B, int64_t ldb, int32_t r,
                                     int32_t with_mean, double *q, const float *d, float *var, float *mean,
                                     void *stream) {
    return row_update<false>("grf_phi_row_condition", phi, f, x, n, col_slot, B, ldb, r, with_mean, q, d, var, mean,
                             stream);
}

extern "C" int grf_phi_row_downdate(const GrfPhi *phi, const float *f, const int32_t *x, int64_t n,
                                    const int32_t *col_slot, const float *B, int64_t ldb, int32_t r,
                                    int32_t with_mean, double *q, const float *d, float *var, float *mean,
                                    void *stream) {
    return row_update<true>("grf_phi_row_downdate", phi, f, x, n, col_slot, B, ldb, r, with_mean, q, d, var, mean,
                            stream);
}
