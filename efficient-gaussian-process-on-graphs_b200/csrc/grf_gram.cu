// Per-length Gram of the training rows for the exact marginal likelihood (grf_b200/mll.py; no reference
// counterpart: the reference estimates the MLL and its gradient by CG and stochastic probes).  With the training ids
// x (n of them, repeats allowed) and the per-length blocks M_0 .. M_{L-1}, stack A[(l, i), c] = M_l[x_i, c]; then
//     E = A A^T,   float64 [L n, L n],   E[l n + i, l' n + j] = <M_l[x_i], M_l'[x_j]>,
// and K(f) = sum_{l, l'} f_l f_l' E[l, :, l', :] + sigma^2 I for every modulator f.
//
// The columns the training rows touch are ranked into slots (PhiBlocks.training_gram, torch).  A slot reached by t_s
// (row, length) entries costs t_s^2 products.  Slots with t_s above a threshold (hub columns) go to a dense float64
// H H^T (cuBLAS through torch); the rest are this file's light kernel, output-stationary:
//
//   gram_light_kernel   one warp per row R = l n + i of E (the rows handed out in descending order of work).  It
//                       walks the light entries of row R in ascending slot; per entry (s, v) its lanes cover the list
//                       of slot s (the (C, v') of every training entry in s) and add v v' into E[R, C] for C >= R.
//                       A __syncwarp separates the entries, so every cell's sum is taken in ascending slot order by
//                       whichever lane holds it, with no atomics; a product of two floats is exact in float64, so only
//                       the sums round.  The warp owns row R, so no other warp writes it.
//   gram_mirror_kernel  E[C, R] = E[R, C] for R < C, by 32 x 32 tiles through shared memory: the (Ln) x (Ln) view of
//                       E is exactly symmetric.

#include "grf_common.cuh"

namespace grf {
namespace {

constexpr int kGramWarps = 8;    // warps per CTA
constexpr int kGramDepth = 4;    // slot-list entries per lane in flight

__global__ void __launch_bounds__(kGramWarps * 32) gram_light_kernel(
    const int32_t *__restrict__ order, int64_t n_rows, const int32_t *__restrict__ row_ptr,
    const int2 *__restrict__ row_ent, const int32_t *__restrict__ slot_ptr, const int2 *__restrict__ slot_ent,
    double *E, int64_t lde) {
    const int lane = threadIdx.x & 31;
    const int64_t warp0 = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    const int64_t n_warps = ((int64_t)gridDim.x * blockDim.x) >> 5;
    for (int64_t u = warp0; u < n_rows; u += n_warps) {
        const int32_t R = order ? __ldg(order + u) : (int32_t)u;
        double *erow = E + (int64_t)R * lde;
        const int32_t kb = __ldg(row_ptr + R), ke = __ldg(row_ptr + R + 1);
        // the next row entry and its slot's list bounds are loaded while the current one is added
        int2 re = make_int2(0, 0);
        int32_t sb = 0, se = 0;
        if (kb < ke) {
            re = __ldg(row_ent + kb);
            sb = __ldg(slot_ptr + re.x);
            se = __ldg(slot_ptr + re.x + 1);
        }
        for (int32_t k = kb; k < ke; ++k) {
            const double v = (double)__int_as_float(re.y);
            const int32_t b = sb, e = se;
            if (k + 1 < ke) {
                re = __ldg(row_ent + k + 1);
                sb = __ldg(slot_ptr + re.x);
                se = __ldg(slot_ptr + re.x + 1);
            }
            for (int32_t t0 = b + lane; t0 < e; t0 += 32 * kGramDepth) {
                int2 ce[kGramDepth];
                double old[kGramDepth];
#pragma unroll
                for (int d = 0; d < kGramDepth; ++d)
                    ce[d] = t0 + 32 * d < e ? __ldg(slot_ent + t0 + 32 * d) : make_int2(-1, 0);
#pragma unroll
                for (int d = 0; d < kGramDepth; ++d)
                    if (ce[d].x >= R) old[d] = erow[ce[d].x];
#pragma unroll
                for (int d = 0; d < kGramDepth; ++d)
                    if (ce[d].x >= R) erow[ce[d].x] = fma(v, (double)__int_as_float(ce[d].y), old[d]);
            }
            __syncwarp();   // the next slot may give this row's cells to other lanes
        }
    }
}

constexpr int kMirrorTile = 32;
constexpr int kMirrorRows = 8;   // thread rows per tile

// block (tc, tr) with tc <= tr: lower tile (tr, tc) <- transpose of upper tile (tc, tr); on the diagonal the reads
// (r <= c) and writes (r > c) are disjoint elements
__global__ void __launch_bounds__(kMirrorTile *kMirrorRows) gram_mirror_kernel(double *E, int64_t N, int64_t lde) {
    __shared__ double tile[kMirrorTile][kMirrorTile + 1];
    const int64_t tc = blockIdx.x, tr = blockIdx.y;
    if (tc > tr) return;
    for (int a = threadIdx.y; a < kMirrorTile; a += kMirrorRows) {
        const int64_t r = tc * kMirrorTile + a, c = tr * kMirrorTile + threadIdx.x;
        if (r < N && c < N && r <= c) tile[a][threadIdx.x] = E[r * lde + c];
    }
    __syncthreads();
    for (int b = threadIdx.y; b < kMirrorTile; b += kMirrorRows) {
        const int64_t r = tr * kMirrorTile + b, c = tc * kMirrorTile + threadIdx.x;
        if (r < N && c < N && r > c) E[r * lde + c] = tile[threadIdx.x][b];
    }
}

}  // namespace
}  // namespace grf

using namespace grf;

extern "C" int grf_gram_light(const int32_t *order, int64_t n_rows, const int32_t *row_ptr, const GrfEntry *row_ent,
                              const int32_t *slot_ptr, const GrfEntry *slot_ent, int64_t n_slots, double *E,
                              int64_t lde, void *stream) {
    GRF_ON_STREAM_DEVICE(stream, E);
    GRF_REQUIRE(n_rows >= 0 && n_slots >= 0 && lde >= n_rows, "grf_gram_light: bad n_rows / n_slots / lde");
    GRF_REQUIRE(n_rows <= INT32_MAX, "grf_gram_light: n_rows exceeds int32");
    if (n_rows == 0) return GRF_OK;
    GRF_REQUIRE(row_ptr && slot_ptr && E, "grf_gram_light: null argument");
    int64_t g = (n_rows + kGramWarps - 1) / kGramWarps;
    if (g > (int64_t)kSmCount * 16) g = (int64_t)kSmCount * 16;
    gram_light_kernel<<<(int)g, kGramWarps * 32, 0, (cudaStream_t)stream>>>(
        order, n_rows, row_ptr, reinterpret_cast<const int2 *>(row_ent), slot_ptr,
        reinterpret_cast<const int2 *>(slot_ent), E, lde);
    return check_cuda(cudaGetLastError(), "gram_light_kernel launch");
}

extern "C" int grf_gram_mirror(double *E, int64_t n_rows, int64_t lde, void *stream) {
    GRF_ON_STREAM_DEVICE(stream, E);
    GRF_REQUIRE(n_rows >= 0 && lde >= n_rows, "grf_gram_mirror: bad n_rows / lde");
    const int64_t tiles = (n_rows + kMirrorTile - 1) / kMirrorTile;
    GRF_REQUIRE(tiles <= 65535, "grf_gram_mirror: n_rows exceeds 65535 tiles of 32");
    if (n_rows == 0) return GRF_OK;
    GRF_REQUIRE(E, "grf_gram_mirror: null argument");
    gram_mirror_kernel<<<dim3((unsigned)tiles, (unsigned)tiles), dim3(kMirrorTile, kMirrorRows), 0,
                         (cudaStream_t)stream>>>(E, n_rows, lde);
    return check_cuda(cudaGetLastError(), "gram_mirror_kernel launch");
}
