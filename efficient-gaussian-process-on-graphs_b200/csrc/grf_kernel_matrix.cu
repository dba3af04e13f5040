// The sparse kernel matrix K = Phi_f Phi_f^T on the device, bit-identical to scipy.
//
// Replaces efficient_graph_gp_sparse/graph_kernels_sparse/fast_grf_kernel_general.py:48-55 of the reference:
//     Phi = csr_matrix((N, N)); Phi += f_p * M_p  (p < min(len(f), L));  return Phi @ Phi.T
// The rules restated here are scipy's (csr_binop_csr for the sum, csr_matmat for the product):
//   Phi_f[r, c]  acc = 0.0; acc = acc + f_p * m over the steps p that store (r, c), ascending p, separate
//                multiply and add (no FMA); explicit zeros of M_p take part; stored iff acc != 0 (NaN is kept)
//   K[i, j]      sums = 0.0; sums = sums + a * Phi_f[j, k] over the entries (k, a) of Phi_f[i] in ascending k;
//                stored iff sums != 0; row i lists its stored j in DESCENDING (first k that touched j, j) order
//                -- the reverse of first-touch order, which is the order scipy's linked list emits
//
// Four stages, each a count / fill pair around a caller scan (grf_scan_counts):
//   1. Phi_f: warp per row, one lane per step segment (lane + 32 s), a warp-min merge of the sorted segments
//   2. Phi_f^T: counting transpose with an atomic cursor per column -- the row order inside a column is
//      arbitrary, which the product allows: the fold runs over k (the outer loop), and inside one k every j
//      occurs once
//   3. row sizes (products per row of K, capped at N) and row bins
//   4. K: a hash of the touched j per row -- warp per row (shared memory), CTA per row (shared memory) or CTA
//      per row with a global-memory table (hub rows), table capacity next_pow2(2 * size) from the row's size.
//      The count pass computes the sums (zero-drop makes the stored count value-dependent) and counts the
//      touched and stored j; the fill pass recomputes them, sorts the stored ones by (first k, j) descending
//      with a bitonic sort and writes them.  The sums need ordering across k, not atomics: the group
//      synchronises after each k.

#include "grf_common.cuh"

namespace grf {

constexpr int kKmatSegPerLane = 4;                   // step segments one lane merges
constexpr int kKmatMaxSteps = 32 * kKmatSegPerLane;  // modulator values used at most (min(len(f), L))
constexpr int kKmatWarpBinMax = 256;                 // row size <= this: warp per row, shared-memory table
constexpr int kKmatCtaBinMax = 2048;                 // ... <= this: CTA per row, shared-memory table
constexpr int kKmatWarpsPerBlock = 4;
constexpr int kKmatCtaThreads = 256;
constexpr int32_t kKmatEmpty = -1;

struct KmatHostF {
    double v[kKmatMaxSteps];
};

// ---------------------------------------------------------------------------------------------------------------
// 1. Phi_f = sum_p f_p M_p from the step-major layout
// ---------------------------------------------------------------------------------------------------------------
template <bool FILL>
__global__ void __launch_bounds__(256) kmat_phi_kernel(const int64_t *__restrict__ off, const int32_t *__restrict__ col,
                                                       const double *__restrict__ val, int64_t n_rows, int32_t n_f,
                                                       KmatHostF fh, const double *__restrict__ fd,
                                                       int32_t *__restrict__ cnt, const int64_t *__restrict__ phi_ptr,
                                                       int32_t *__restrict__ phi_col, double *__restrict__ phi_val) {
    const int lane = threadIdx.x & 31;
    const int64_t warp0 = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    const int64_t nwarps = ((int64_t)gridDim.x * blockDim.x) >> 5;
    double fs[kKmatSegPerLane];
#pragma unroll
    for (int s = 0; s < kKmatSegPerLane; ++s) {
        const int p = lane + 32 * s;
        fs[s] = p < n_f ? (fd ? fd[p] : fh.v[p]) : 0.0;
    }
    for (int64_t r = warp0; r < n_rows; r += nwarps) {
        int64_t pos[kKmatSegPerLane], end[kKmatSegPerLane];
        int32_t head[kKmatSegPerLane];
#pragma unroll
        for (int s = 0; s < kKmatSegPerLane; ++s) {
            const int p = lane + 32 * s;
            pos[s] = end[s] = 0;
            if (p < n_f) {
                pos[s] = off[(int64_t)p * n_rows + r];
                end[s] = off[(int64_t)p * n_rows + r + 1];
            }
            head[s] = pos[s] < end[s] ? col[pos[s]] : INT32_MAX;
        }
        const int64_t out = FILL ? phi_ptr[r] : 0;
        int32_t n = 0;
        for (;;) {
            int32_t m = head[0];
#pragma unroll
            for (int s = 1; s < kKmatSegPerLane; ++s) m = min(m, head[s]);
#pragma unroll
            for (int d = 16; d > 0; d >>= 1) m = min(m, __shfl_xor_sync(0xffffffffu, m, d));
            if (m == INT32_MAX) break;
            // fold the steps that store column m in ascending p = lane + 32 s: s outer, lanes inner
            double acc = 0.0;
#pragma unroll
            for (int s = 0; s < kKmatSegPerLane; ++s) {
                const bool hit = head[s] == m;
                const double term = hit ? __dmul_rn(fs[s], val[pos[s]]) : 0.0;
                unsigned mask = __ballot_sync(0xffffffffu, hit);
                while (mask) {
                    const int l = __ffs(mask) - 1;
                    acc = __dadd_rn(acc, __shfl_sync(0xffffffffu, term, l));
                    mask &= mask - 1;
                }
                if (hit) {
                    ++pos[s];
                    head[s] = pos[s] < end[s] ? col[pos[s]] : INT32_MAX;
                }
            }
            if (acc != 0.0) {  // csr_binop_csr drops exact zeros; NaN != 0 is kept
                if (FILL && lane == 0) {
                    phi_col[out + n] = m;
                    phi_val[out + n] = acc;
                }
                ++n;
            }
        }
        if (!FILL && lane == 0) cnt[r] = n;
    }
}

// ---------------------------------------------------------------------------------------------------------------
// 2. Phi_f^T by counting transpose
// ---------------------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256) kmat_tcount_kernel(const int64_t *__restrict__ phi_ptr,
                                                          const int32_t *__restrict__ phi_col, int64_t n_rows,
                                                          int32_t *__restrict__ tcnt) {
    const int lane = threadIdx.x & 31;
    const int64_t warp0 = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    const int64_t nwarps = ((int64_t)gridDim.x * blockDim.x) >> 5;
    for (int64_t r = warp0; r < n_rows; r += nwarps)
        for (int64_t i = phi_ptr[r] + lane; i < phi_ptr[r + 1]; i += 32) atomicAdd(&tcnt[phi_col[i]], 1);
}

__global__ void __launch_bounds__(256) kmat_tcursor_kernel(const int64_t *__restrict__ tptr, int64_t n_cols,
                                                           unsigned long long *__restrict__ cursor) {
    for (int64_t c = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; c < n_cols; c += (int64_t)gridDim.x * blockDim.x)
        cursor[c] = (unsigned long long)tptr[c];
}

__global__ void __launch_bounds__(256) kmat_tfill_kernel(const int64_t *__restrict__ phi_ptr,
                                                         const int32_t *__restrict__ phi_col,
                                                         const double *__restrict__ phi_val, int64_t n_rows,
                                                         unsigned long long *__restrict__ cursor,
                                                         int32_t *__restrict__ trow, double *__restrict__ tval) {
    const int lane = threadIdx.x & 31;
    const int64_t warp0 = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    const int64_t nwarps = ((int64_t)gridDim.x * blockDim.x) >> 5;
    for (int64_t r = warp0; r < n_rows; r += nwarps)
        for (int64_t i = phi_ptr[r] + lane; i < phi_ptr[r + 1]; i += 32) {
            const int64_t at = (int64_t)atomicAdd(&cursor[phi_col[i]], 1ull);
            trow[at] = (int32_t)r;
            tval[at] = phi_val[i];
        }
}

// ---------------------------------------------------------------------------------------------------------------
// 3. row sizes and bins
// ---------------------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256) kmat_size_kernel(const int64_t *__restrict__ phi_ptr,
                                                        const int32_t *__restrict__ phi_col,
                                                        const int64_t *__restrict__ tptr, int64_t n_rows,
                                                        int32_t *__restrict__ size) {
    const int lane = threadIdx.x & 31;
    const int64_t warp0 = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    const int64_t nwarps = ((int64_t)gridDim.x * blockDim.x) >> 5;
    for (int64_t r = warp0; r < n_rows; r += nwarps) {
        int64_t s = 0;
        for (int64_t i = phi_ptr[r] + lane; i < phi_ptr[r + 1]; i += 32) {
            const int32_t k = phi_col[i];
            s += tptr[k + 1] - tptr[k];
        }
#pragma unroll
        for (int d = 16; d > 0; d >>= 1) s += __shfl_xor_sync(0xffffffffu, s, d);
        if (lane == 0) size[r] = (int32_t)(s < n_rows ? s : n_rows);
    }
}

__host__ __device__ __forceinline__ int kmat_bin_of(int32_t size) {
    return size <= kKmatWarpBinMax ? 0 : size <= kKmatCtaBinMax ? 1 : 2;
}

__global__ void __launch_bounds__(256) kmat_bin_kernel(const int32_t *__restrict__ size, int64_t n_rows,
                                                       int32_t *__restrict__ rows, unsigned long long *__restrict__ stats) {
    for (int64_t r = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; r < n_rows; r += (int64_t)gridDim.x * blockDim.x) {
        const int32_t s = size[r];
        const int b = kmat_bin_of(s);
        const unsigned long long at = atomicAdd(&stats[b], 1ull);
        rows[(int64_t)b * n_rows + (int64_t)at] = (int32_t)r;
        if (b == 2) atomicMax(&stats[3], (unsigned long long)s);
    }
}

// ---------------------------------------------------------------------------------------------------------------
// 4. K = Phi_f Phi_f^T
// ---------------------------------------------------------------------------------------------------------------
// One group's table for rows of size <= max_size: capacity next_pow2(2 * max_size) slots, a list of the claimed
// slots (touched j, at most max_size) and the sort buffer of the stored ones.
struct KmatSlice {
    double *sums;
    unsigned long long *skey;
    double *sval;
    int32_t *keys;
    int32_t *first;
    int32_t *list;
    uint32_t cap_max;
};

__host__ __device__ __forceinline__ int64_t kmat_slice_bytes(int32_t max_size) {
    const int64_t m = max_size < 1 ? 1 : max_size;
    const int64_t cap = next_pow2((uint32_t)(2 * m)), srt = next_pow2((uint32_t)m);
    const int64_t bytes = cap * 8 + srt * 16 + cap * 8 + m * 4;
    return (bytes + 15) & ~(int64_t)15;
}

__device__ __forceinline__ KmatSlice kmat_carve(unsigned char *base, int32_t max_size) {
    const int64_t m = max_size < 1 ? 1 : max_size;
    const int64_t cap = next_pow2((uint32_t)(2 * m)), srt = next_pow2((uint32_t)m);
    KmatSlice t;
    t.sums = (double *)base;
    t.skey = (unsigned long long *)(t.sums + cap);
    t.sval = (double *)(t.skey + srt);
    t.keys = (int32_t *)(t.sval + srt);
    t.first = t.keys + cap;
    t.list = t.first + cap;
    t.cap_max = (uint32_t)cap;
    return t;
}

template <bool WARP>
__device__ __forceinline__ void kmat_sync() {
    if (WARP)
        __syncwarp();
    else
        __syncthreads();
}

struct KmatOps {
    const int64_t *phi_ptr;
    const int32_t *phi_col;
    const double *phi_val;
    const int64_t *tptr;
    const int32_t *trow;
    const double *tval;
    const int32_t *size;
    int32_t *touched;  // count pass
    int32_t *stored;   // count pass
    const int64_t *kptr;  // fill pass
    int32_t *kcol;
    double *kval;
    int32_t *overflow;
};

// Row r of K on one group (a warp or a CTA) that owns table t; gcnt: two shared ints of the group.
template <bool FILL, bool WARP>
__device__ void kmat_row(const KmatOps &o, int64_t r, const KmatSlice &t, int *gcnt, int rank, int G) {
    const int32_t size = o.size[r];
    const uint32_t cap = next_pow2(2u * (uint32_t)(size < 1 ? 1 : size));
    const int shift = 32 - (bit_width(cap) - 1);
    bool over = cap > t.cap_max;
    if (rank == 0) gcnt[0] = gcnt[1] = 0;
    kmat_sync<WARP>();
    const int64_t b = o.phi_ptr[r], e = o.phi_ptr[r + 1];
    if (!over) {
        for (int64_t p = b; p < e; ++p) {
            const int32_t k = o.phi_col[p];
            const double a = o.phi_val[p];
            const int64_t te = o.tptr[k + 1];
            for (int64_t q = o.tptr[k] + rank; q < te; q += G) {
                const int32_t j = o.trow[q];
                const double prod = __dmul_rn(a, o.tval[q]);
                uint32_t h = ((uint32_t)j * 2654435761u) >> shift;
                for (uint32_t probe = 0;; ++probe) {
                    if (probe == cap) {  // cannot happen while size >= the row's touched count
                        over = true;
                        break;
                    }
                    const int32_t prev = atomicCAS(&t.keys[h], kKmatEmpty, j);
                    if (prev == kKmatEmpty) {  // first touch of j: at this k, by this thread only
                        t.first[h] = (int32_t)(p - b);
                        t.sums[h] = __dadd_rn(0.0, prod);
                        const int at = atomicAdd(&gcnt[0], 1);
                        if (at < size)
                            t.list[at] = (int32_t)h;
                        else
                            over = true;
                        break;
                    }
                    if (prev == j) {  // j occurs once per k: no other thread adds to this slot now
                        t.sums[h] = __dadd_rn(t.sums[h], prod);
                        break;
                    }
                    h = (h + 1) & (cap - 1);
                }
            }
            kmat_sync<WARP>();  // the next k adds after this one
        }
    }
    const int nt = min(gcnt[0], size);
    if (!FILL) {
        int mine = 0;
        for (int u = rank; u < nt; u += G) mine += t.sums[t.list[u]] != 0.0;
        if (mine) atomicAdd(&gcnt[1], mine);
        kmat_sync<WARP>();
        if (rank == 0) {
            o.touched[r] = gcnt[0];
            o.stored[r] = gcnt[1];
        }
    } else {
        for (int u = rank; u < nt; u += G) {
            const int32_t h = t.list[u];
            const double s = t.sums[h];
            if (s != 0.0) {
                const int at = atomicAdd(&gcnt[1], 1);
                t.skey[at] = (((unsigned long long)(uint32_t)t.first[h] << 32) | (uint32_t)t.keys[h]) + 1ull;
                t.sval[at] = s;
            }
        }
        kmat_sync<WARP>();
        const int ns = gcnt[1];
        const int64_t out = o.kptr[r];
        if (o.kptr[r + 1] - out != ns) {
            over = true;
        } else if (ns > 0) {
            const int n2 = (int)next_pow2((uint32_t)ns);
            for (int u = ns + rank; u < n2; u += G) t.skey[u] = 0ull;  // padding sorts last
            kmat_sync<WARP>();
            // bitonic sort, descending by (first k, j) + 1
            for (int kk = 2; kk <= n2; kk <<= 1) {
                for (int jj = kk >> 1; jj > 0; jj >>= 1) {
                    for (int i = rank; i < n2; i += G) {
                        const int ix = i ^ jj;
                        if (ix > i) {
                            const unsigned long long x = t.skey[i], y = t.skey[ix];
                            const bool desc = (i & kk) == 0;
                            if (desc ? x < y : x > y) {
                                t.skey[i] = y;
                                t.skey[ix] = x;
                                const double vx = t.sval[i];
                                t.sval[i] = t.sval[ix];
                                t.sval[ix] = vx;
                            }
                        }
                    }
                    kmat_sync<WARP>();
                }
            }
            for (int u = rank; u < ns; u += G) {
                o.kcol[out + u] = (int32_t)(uint32_t)((t.skey[u] - 1ull) & 0xffffffffull);
                o.kval[out + u] = t.sval[u];
            }
        }
    }
    for (int u = rank; u < nt; u += G) t.keys[t.list[u]] = kKmatEmpty;  // leave the table empty for the next row
    if (over) atomicExch(o.overflow, 1);
    kmat_sync<WARP>();
}

template <bool FILL>
__global__ void __launch_bounds__(32 * kKmatWarpsPerBlock) kmat_rows_warp_kernel(KmatOps o, const int32_t *rows,
                                                                                 int64_t n) {
    extern __shared__ __align__(16) unsigned char kmat_smem[];
    __shared__ int gcnt[kKmatWarpsPerBlock][2];
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const KmatSlice t = kmat_carve(kmat_smem + warp * kmat_slice_bytes(kKmatWarpBinMax), kKmatWarpBinMax);
    for (uint32_t u = lane; u < t.cap_max; u += 32) t.keys[u] = kKmatEmpty;
    __syncwarp();
    for (int64_t i = (int64_t)blockIdx.x * kKmatWarpsPerBlock + warp; i < n; i += (int64_t)gridDim.x * kKmatWarpsPerBlock)
        kmat_row<FILL, true>(o, rows[i], t, gcnt[warp], lane, 32);
}

template <bool FILL>
__device__ __forceinline__ void kmat_rows_cta(const KmatOps &o, const int32_t *rows, int64_t n, const KmatSlice &t) {
    __shared__ int gcnt[2];
    for (uint32_t u = threadIdx.x; u < t.cap_max; u += blockDim.x) t.keys[u] = kKmatEmpty;
    __syncthreads();
    for (int64_t i = blockIdx.x; i < n; i += gridDim.x) kmat_row<FILL, false>(o, rows[i], t, gcnt, threadIdx.x, blockDim.x);
}

template <bool FILL>
__global__ void __launch_bounds__(kKmatCtaThreads) kmat_rows_cta_kernel(KmatOps o, const int32_t *rows, int64_t n) {
    extern __shared__ __align__(16) unsigned char kmat_smem[];
    kmat_rows_cta<FILL>(o, rows, n, kmat_carve(kmat_smem, kKmatCtaBinMax));
}

// hub rows: the same CTA-per-row code on a table in global memory (slice blockIdx.x of the workspace)
template <bool FILL>
__global__ void __launch_bounds__(kKmatCtaThreads) kmat_rows_global_kernel(KmatOps o, const int32_t *rows, int64_t n,
                                                                           unsigned char *ws, int32_t max_size) {
    kmat_rows_cta<FILL>(o, rows, n, kmat_carve(ws + blockIdx.x * kmat_slice_bytes(max_size), max_size));
}

static inline int kmat_grid(int64_t items, int per_block, int64_t cap) {
    int64_t g = (items + per_block - 1) / per_block;
    if (g > cap) g = cap;
    if (g < 1) g = 1;
    return (int)g;
}

// The shared-memory bins need more than the default 48 KB: opt in once per (device, kernel).
constexpr int kKmatMaxDevices = 64;
static bool g_kmat_smem_set[kKmatMaxDevices][4];

template <typename K>
static int kmat_smem_opt_in(K kern, int which, size_t smem) {
    int dev = 0;
    GRF_CUDA_OK(cudaGetDevice(&dev));
    if (dev >= 0 && dev < kKmatMaxDevices && g_kmat_smem_set[dev][which]) return GRF_OK;
    GRF_CUDA_OK(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    if (dev >= 0 && dev < kKmatMaxDevices) g_kmat_smem_set[dev][which] = true;  // idempotent: a race only repeats it
    return GRF_OK;
}

template <bool FILL>
static int kmat_launch(const KmatOps &o, int64_t n_rows, const int32_t *rows, const int64_t *bin_rows,
                       int32_t max_size, int32_t global_ctas, void *workspace, cudaStream_t st) {
    GRF_CUDA_OK(cudaMemsetAsync(o.overflow, 0, sizeof(int32_t), st));
    if (bin_rows[0] > 0) {
        const size_t smem = (size_t)kKmatWarpsPerBlock * kmat_slice_bytes(kKmatWarpBinMax);
        const int rc = kmat_smem_opt_in(kmat_rows_warp_kernel<FILL>, FILL ? 1 : 0, smem);
        if (rc != GRF_OK) return rc;
        kmat_rows_warp_kernel<FILL><<<kmat_grid(bin_rows[0], kKmatWarpsPerBlock, (int64_t)kSmCount * 8),
                                      32 * kKmatWarpsPerBlock, smem, st>>>(o, rows, bin_rows[0]);
        GRF_CUDA_OK(cudaGetLastError());
    }
    if (bin_rows[1] > 0) {
        const size_t smem = (size_t)kmat_slice_bytes(kKmatCtaBinMax);
        const int rc = kmat_smem_opt_in(kmat_rows_cta_kernel<FILL>, FILL ? 3 : 2, smem);
        if (rc != GRF_OK) return rc;
        kmat_rows_cta_kernel<FILL><<<kmat_grid(bin_rows[1], 1, (int64_t)kSmCount * 2), kKmatCtaThreads, smem, st>>>(
            o, rows + n_rows, bin_rows[1]);
        GRF_CUDA_OK(cudaGetLastError());
    }
    if (bin_rows[2] > 0) {
        kmat_rows_global_kernel<FILL><<<global_ctas, kKmatCtaThreads, 0, st>>>(o, rows + 2 * n_rows, bin_rows[2],
                                                                              (unsigned char *)workspace, max_size);
        GRF_CUDA_OK(cudaGetLastError());
    }
    return GRF_OK;
}

}  // namespace grf

using namespace grf;

static int kmat_phi_args(const int64_t *offsets, const int32_t *col, const double *val, int64_t n_rows,
                         int32_t n_steps, const double *f, int32_t n_f, int32_t f_on_host, const char *who) {
    GRF_REQUIRE(n_rows >= 0 && n_steps >= 1 && n_f >= 0, "%s: bad shape", who);
    GRF_REQUIRE(n_f <= n_steps, "%s: n_f = %d exceeds n_steps = %d (pass min(len(f), L))", who, n_f, n_steps);
    if (n_f > kKmatMaxSteps)
        return fail(GRF_ERR_UNSUPPORTED, "%s: at most %d modulator values are merged, got %d", who, kKmatMaxSteps, n_f);
    GRF_REQUIRE(f_on_host == 0 || f_on_host == 1, "%s: f_on_host must be 0 (device f) or 1 (host f)", who);
    GRF_REQUIRE(n_f == 0 || f, "%s: null f", who);
    GRF_REQUIRE(n_rows == 0 || (offsets && col && val), "%s: null buffer", who);
    return GRF_OK;
}

static void kmat_host_f(const double *f, int32_t n_f, int32_t f_on_host, KmatHostF &fh, const double *&fd) {
    for (int p = 0; p < kKmatMaxSteps; ++p) fh.v[p] = 0.0;
    fd = nullptr;
    if (f_on_host) {
        for (int p = 0; p < n_f; ++p) fh.v[p] = f[p];
    } else {
        fd = f;
    }
}

extern "C" int grf_kmat_phi_count(const int64_t *offsets_step_major, const int32_t *col, const double *val,
                                  int64_t n_rows, int32_t n_steps, const double *f, int32_t n_f, int32_t f_on_host,
                                  int32_t *phi_cnt, void *stream) {
    GRF_ON_STREAM_DEVICE(stream, phi_cnt);
    int rc = kmat_phi_args(offsets_step_major, col, val, n_rows, n_steps, f, n_f, f_on_host, "grf_kmat_phi_count");
    if (rc != GRF_OK) return rc;
    if (n_rows == 0) return GRF_OK;
    GRF_REQUIRE(phi_cnt, "grf_kmat_phi_count: null phi_cnt");
    KmatHostF fh;
    const double *fd;
    kmat_host_f(f, n_f, f_on_host, fh, fd);
    kmat_phi_kernel<false><<<kmat_grid(n_rows, 8, (int64_t)kSmCount * 32), 256, 0, (cudaStream_t)stream>>>(
        offsets_step_major, col, val, n_rows, n_f, fh, fd, phi_cnt, nullptr, nullptr, nullptr);
    return check_cuda(cudaGetLastError(), "kmat_phi_kernel<count> launch");
}

extern "C" int grf_kmat_phi_fill(const int64_t *offsets_step_major, const int32_t *col, const double *val,
                                 int64_t n_rows, int32_t n_steps, const double *f, int32_t n_f, int32_t f_on_host,
                                 const int64_t *phi_ptr, int32_t *phi_col, double *phi_val, void *stream) {
    GRF_ON_STREAM_DEVICE(stream, phi_ptr);
    int rc = kmat_phi_args(offsets_step_major, col, val, n_rows, n_steps, f, n_f, f_on_host, "grf_kmat_phi_fill");
    if (rc != GRF_OK) return rc;
    if (n_rows == 0) return GRF_OK;
    GRF_REQUIRE(phi_ptr, "grf_kmat_phi_fill: null phi_ptr");
    KmatHostF fh;
    const double *fd;
    kmat_host_f(f, n_f, f_on_host, fh, fd);
    kmat_phi_kernel<true><<<kmat_grid(n_rows, 8, (int64_t)kSmCount * 32), 256, 0, (cudaStream_t)stream>>>(
        offsets_step_major, col, val, n_rows, n_f, fh, fd, nullptr, phi_ptr, phi_col, phi_val);
    return check_cuda(cudaGetLastError(), "kmat_phi_kernel<fill> launch");
}

extern "C" int grf_kmat_transpose_count(const int64_t *phi_ptr, const int32_t *phi_col, int64_t n_rows,
                                        int64_t n_cols, int32_t *tcnt, void *stream) {
    GRF_ON_STREAM_DEVICE(stream, tcnt);
    GRF_REQUIRE(n_rows >= 0 && n_cols >= 0 && n_rows < (1ll << 31) && n_cols < (1ll << 31),
                "grf_kmat_transpose_count: bad shape");
    if (n_cols == 0) return GRF_OK;
    GRF_REQUIRE(tcnt && (n_rows == 0 || (phi_ptr && phi_col)), "grf_kmat_transpose_count: null buffer");
    cudaStream_t st = (cudaStream_t)stream;
    GRF_CUDA_OK(cudaMemsetAsync(tcnt, 0, (size_t)n_cols * sizeof(int32_t), st));
    if (n_rows == 0) return GRF_OK;
    kmat_tcount_kernel<<<kmat_grid(n_rows, 8, (int64_t)kSmCount * 32), 256, 0, st>>>(phi_ptr, phi_col, n_rows, tcnt);
    return check_cuda(cudaGetLastError(), "kmat_tcount_kernel launch");
}

extern "C" int grf_kmat_transpose_fill(const int64_t *phi_ptr, const int32_t *phi_col, const double *phi_val,
                                       int64_t n_rows, int64_t n_cols, const int64_t *tptr, int64_t *cursor,
                                       int32_t *trow, double *tval, void *stream) {
    GRF_ON_STREAM_DEVICE(stream, tptr);
    GRF_REQUIRE(n_rows >= 0 && n_cols >= 0 && n_rows < (1ll << 31) && n_cols < (1ll << 31),
                "grf_kmat_transpose_fill: bad shape");
    if (n_rows == 0 || n_cols == 0) return GRF_OK;
    GRF_REQUIRE(phi_ptr && phi_col && phi_val && tptr && cursor, "grf_kmat_transpose_fill: null buffer");
    cudaStream_t st = (cudaStream_t)stream;
    kmat_tcursor_kernel<<<kmat_grid(n_cols, 256, (int64_t)kSmCount * 16), 256, 0, st>>>(
        tptr, n_cols, (unsigned long long *)cursor);
    GRF_CUDA_OK(cudaGetLastError());
    kmat_tfill_kernel<<<kmat_grid(n_rows, 8, (int64_t)kSmCount * 32), 256, 0, st>>>(
        phi_ptr, phi_col, phi_val, n_rows, (unsigned long long *)cursor, trow, tval);
    return check_cuda(cudaGetLastError(), "kmat_tfill_kernel launch");
}

extern "C" int grf_kmat_row_sizes(const int64_t *phi_ptr, const int32_t *phi_col, const int64_t *tptr, int64_t n_rows,
                                  int32_t *size, void *stream) {
    GRF_ON_STREAM_DEVICE(stream, size);
    GRF_REQUIRE(n_rows >= 0 && n_rows < (1ll << 31), "grf_kmat_row_sizes: bad shape");
    if (n_rows == 0) return GRF_OK;
    GRF_REQUIRE(phi_ptr && phi_col && tptr && size, "grf_kmat_row_sizes: null buffer");
    kmat_size_kernel<<<kmat_grid(n_rows, 8, (int64_t)kSmCount * 32), 256, 0, (cudaStream_t)stream>>>(
        phi_ptr, phi_col, tptr, n_rows, size);
    return check_cuda(cudaGetLastError(), "kmat_size_kernel launch");
}

extern "C" int grf_kmat_bin(const int32_t *size, int64_t n_rows, int32_t *rows, int64_t *stats, void *stream) {
    GRF_ON_STREAM_DEVICE(stream, stats);
    GRF_REQUIRE(n_rows >= 0 && n_rows < (1ll << 31), "grf_kmat_bin: bad shape");
    GRF_REQUIRE(stats, "grf_kmat_bin: null stats");
    cudaStream_t st = (cudaStream_t)stream;
    GRF_CUDA_OK(cudaMemsetAsync(stats, 0, 4 * sizeof(int64_t), st));
    if (n_rows == 0) return GRF_OK;
    GRF_REQUIRE(size && rows, "grf_kmat_bin: null buffer");
    kmat_bin_kernel<<<kmat_grid(n_rows, 256, (int64_t)kSmCount * 16), 256, 0, st>>>(size, n_rows, rows,
                                                                                   (unsigned long long *)stats);
    return check_cuda(cudaGetLastError(), "kmat_bin_kernel launch");
}

extern "C" int64_t grf_kmat_workspace_bytes(int32_t max_size, int32_t global_ctas) {
    if (global_ctas <= 0 || max_size <= kKmatCtaBinMax) return 0;
    return (int64_t)global_ctas * kmat_slice_bytes(max_size);
}

static int kmat_common_args(const int64_t *phi_ptr, const int32_t *phi_col, const double *phi_val,
                            const int64_t *tptr, const int32_t *trow, const double *tval, int64_t n_rows,
                            const int32_t *size, const int32_t *rows, const int64_t *bin_rows, int32_t max_size,
                            int32_t global_ctas, void *workspace, int64_t workspace_bytes, int32_t *overflow,
                            const char *who) {
    GRF_REQUIRE(n_rows >= 0 && n_rows < (1ll << 30), "%s: bad shape", who);
    GRF_REQUIRE(bin_rows, "%s: null bin_rows", who);
    GRF_REQUIRE(bin_rows[0] >= 0 && bin_rows[1] >= 0 && bin_rows[2] >= 0 &&
                    bin_rows[0] + bin_rows[1] + bin_rows[2] <= n_rows,
                "%s: bad bin_rows", who);
    if (n_rows == 0) return GRF_OK;
    GRF_REQUIRE(phi_ptr && phi_col && phi_val && tptr && trow && tval && size && rows && overflow,
                "%s: null buffer", who);
    if (bin_rows[2] > 0) {
        GRF_REQUIRE(max_size > kKmatCtaBinMax && max_size <= n_rows, "%s: max_size %d outside the global bin", who,
                    max_size);
        GRF_REQUIRE(global_ctas >= 1, "%s: global_ctas must be >= 1", who);
        GRF_REQUIRE(workspace && workspace_bytes >= grf_kmat_workspace_bytes(max_size, global_ctas),
                    "%s: workspace of %lld bytes, need %lld", who, (long long)workspace_bytes,
                    (long long)grf_kmat_workspace_bytes(max_size, global_ctas));
    }
    return GRF_OK;
}

extern "C" int grf_kmat_count(const int64_t *phi_ptr, const int32_t *phi_col, const double *phi_val,
                              const int64_t *tptr, const int32_t *trow, const double *tval, int64_t n_rows,
                              const int32_t *size, const int32_t *rows, const int64_t *bin_rows, int32_t max_size,
                              int32_t global_ctas, void *workspace, int64_t workspace_bytes, int32_t *touched,
                              int32_t *stored, int32_t *overflow, void *stream) {
    GRF_ON_STREAM_DEVICE(stream, phi_ptr);
    int rc = kmat_common_args(phi_ptr, phi_col, phi_val, tptr, trow, tval, n_rows, size, rows, bin_rows, max_size,
                              global_ctas, workspace, workspace_bytes, overflow, "grf_kmat_count");
    if (rc != GRF_OK) return rc;
    if (n_rows == 0) return GRF_OK;
    GRF_REQUIRE(touched && stored, "grf_kmat_count: null counts");
    KmatOps o{phi_ptr, phi_col, phi_val, tptr, trow, tval, size, touched, stored, nullptr, nullptr, nullptr, overflow};
    return kmat_launch<false>(o, n_rows, rows, bin_rows, max_size, global_ctas, workspace, (cudaStream_t)stream);
}

extern "C" int grf_kmat_fill(const int64_t *phi_ptr, const int32_t *phi_col, const double *phi_val,
                             const int64_t *tptr, const int32_t *trow, const double *tval, int64_t n_rows,
                             const int32_t *size, const int32_t *rows, const int64_t *bin_rows, int32_t max_size,
                             int32_t global_ctas, void *workspace, int64_t workspace_bytes, const int64_t *kptr,
                             int32_t *kcol, double *kval, int32_t *overflow, void *stream) {
    GRF_ON_STREAM_DEVICE(stream, phi_ptr);
    int rc = kmat_common_args(phi_ptr, phi_col, phi_val, tptr, trow, tval, n_rows, size, rows, bin_rows, max_size,
                              global_ctas, workspace, workspace_bytes, overflow, "grf_kmat_fill");
    if (rc != GRF_OK) return rc;
    if (n_rows == 0) return GRF_OK;
    GRF_REQUIRE(kptr, "grf_kmat_fill: null kptr");
    KmatOps o{phi_ptr, phi_col, phi_val, tptr, trow, tval, size, nullptr, nullptr, kptr, kcol, kval, overflow};
    return kmat_launch<true>(o, n_rows, rows, bin_rows, max_size, global_ctas, workspace, (cudaStream_t)stream);
}
