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
