/*
 * Coupled walk draws in plain C (TEST INFRASTRUCTURE ONLY -- see oracle/__init__.py): the bit-level answer of
 * grf_walk with GRF_DRAW_COUPLE_* bits in draw_mode (definitions at GrfWalkCfg.seed in include/grf_b200.h).
 *
 * Compiled into its own library together with oracle/grf_oracle.c, whose Philox, record sort, result type and
 * accessors (grf_oracle_nnz / _visits / _copy / _free) it reuses unchanged; the independent-draws oracle is not
 * touched.  Per start node all W walks advance one step at a time and every length's visits are recorded in
 * walk order, then merged exactly as grf_oracle_build merges them.
 */
#include "grf_oracle.c"

/*
 * Coupled draws (GRF_DRAW_COUPLE_* in include/grf_b200.h; native Philox draws only): the W walks of a start
 * node advance one step at a time.  coupling bit 2 = antithetic termination (walk 2q+1 halts on walk 2q's
 * halting word XOR 0x80000000), bit 4 = repelling neighbours (the m walks of the start node that stand on v,
 * still walk and do not halt, ranked j in walk order, take (c + floor(j * deg / m)) mod deg with
 * c = (U * deg) >> 32, U = word 0 of philox(start, v, step, 1)).  Visits are summed as in grf_oracle_build.
 */
GrfOracleResult *grf_oracle_build_coupled(int64_t n_nodes, const int32_t *indptr, const int32_t *indices,
                                          const double *data, int64_t start_lo, int64_t start_hi, int32_t W, int32_t L,
                                          double p_halt, int32_t coupling, uint64_t seed, int32_t load_mode,
                                          int32_t scale_mode) {
    (void)n_nodes;
    GrfOracleResult *r = (GrfOracleResult *)calloc(1, sizeof(*r));
    int64_t n_local = start_hi - start_lo;
    r->n_local = n_local;
    r->L = L;
    r->nnz = (int64_t *)calloc((size_t)L, sizeof(int64_t));
    r->cap = (int64_t *)calloc((size_t)L, sizeof(int64_t));
    r->indptr = (int64_t **)calloc((size_t)L, sizeof(int64_t *));
    r->indices = (int32_t **)calloc((size_t)L, sizeof(int32_t *));
    r->data = (double **)calloc((size_t)L, sizeof(double *));
    for (int s = 0; s < L; ++s) r->indptr[s] = (int64_t *)calloc((size_t)n_local + 1, sizeof(int64_t));

    Rec *recs = (Rec *)malloc((size_t)W * sizeof(Rec));
    int32_t *cur = (int32_t *)malloc((size_t)W * sizeof(int32_t)); /* -1 = stopped */
    double *load = (double *)malloc((size_t)W * sizeof(double));
    int32_t *cont = (int32_t *)malloc((size_t)W * sizeof(int32_t));
    int32_t *rank = (int32_t *)malloc((size_t)W * sizeof(int32_t));
    int32_t *count = (int32_t *)malloc((size_t)W * sizeof(int32_t));
    const double one_minus_p = 1.0 - p_halt;
    double thr = floor(p_halt * 4294967296.0);
    if (thr < 0) thr = 0;
    if (thr > 4294967296.0) thr = 4294967296.0;
    const uint64_t halt_thr = (uint64_t)thr;
    const uint32_t key[2] = {(uint32_t)seed, (uint32_t)(seed >> 32)};
    const double recip = 1.0 / (double)W;

    for (int64_t start = start_lo; start < start_hi; ++start) {
        const int64_t row = start - start_lo;
        for (int32_t w = 0; w < W; ++w) {
            cur[w] = (int32_t)start;
            load[w] = 1.0;
        }
        for (int32_t step = 0; step < L; ++step) {
            /* the visits of this length, in walk order, merged per node */
            int32_t n = 0;
            for (int32_t w = 0; w < W; ++w) {
                if (cur[w] < 0) continue;
                recs[n].node = cur[w];
                recs[n].seq = w;
                recs[n].load = load[w];
                ++n;
            }
            r->visits += n;
            qsort(recs, (size_t)n, sizeof(Rec), rec_cmp);
            int32_t i = 0;
            while (i < n) {
                volatile double sum = 0.0;
                int32_t j = i;
                while (j < n && recs[j].node == recs[i].node) {
                    sum = sum + recs[j].load;
                    ++j;
                }
                double v = sum;
                v = scale_mode == 0 ? v * recip : v / (double)W;
                push_entry(r, step, recs[i].node, v);
                i = j;
            }
            r->indptr[step][row + 1] = r->nnz[step];
            if (step == L - 1) break;
            /* halting decisions */
            for (int32_t w = 0; w < W; ++w) {
                cont[w] = 0;
                if (cur[w] < 0) continue;
                const int32_t deg = indptr[cur[w] + 1] - indptr[cur[w]];
                if (deg == 0) continue;
                const int32_t src = ((coupling & 2) && (w & 1)) ? w - 1 : w;
                const uint64_t gid = (uint64_t)start * (uint64_t)W + (uint64_t)src;
                const uint32_t ctr[4] = {(uint32_t)gid, (uint32_t)(gid >> 32), (uint32_t)(step >> 1), 0u};
                uint32_t x[4];
                grf_oracle_philox(ctr, key, x);
                uint32_t xh = x[2 * (step & 1)];
                if (src != w) xh ^= 0x80000000u;
                cont[w] = (uint64_t)xh >= halt_thr;
            }
            /* repelling: rank and count of the continuing walks per node (recs is sorted by (node, walk)) */
            if (coupling & 4) {
                i = 0;
                while (i < n) {
                    int32_t j = i, m = 0;
                    while (j < n && recs[j].node == recs[i].node) {
                        if (cont[recs[j].seq]) rank[recs[j].seq] = m++;
                        ++j;
                    }
                    for (int32_t q = i; q < j; ++q) count[recs[q].seq] = m;
                    i = j;
                }
            }
            /* the moves */
            for (int32_t w = 0; w < W; ++w) {
                if (!cont[w]) {
                    cur[w] = -1;
                    continue;
                }
                const int32_t s = indptr[cur[w]];
                const int32_t deg = indptr[cur[w] + 1] - s;
                int32_t k;
                if (coupling & 4) {
                    const uint32_t ctr[4] = {(uint32_t)start, (uint32_t)cur[w], (uint32_t)step, 1u};
                    uint32_t x[4];
                    grf_oracle_philox(ctr, key, x);
                    const uint64_t c = ((uint64_t)x[0] * (uint64_t)(uint32_t)deg) >> 32;
                    k = (int32_t)((c + (uint64_t)rank[w] * (uint64_t)deg / (uint64_t)count[w]) % (uint64_t)deg);
                } else {
                    const uint64_t gid = (uint64_t)start * (uint64_t)W + (uint64_t)w;
                    const uint32_t ctr[4] = {(uint32_t)gid, (uint32_t)(gid >> 32), (uint32_t)(step >> 1), 0u};
                    uint32_t x[4];
                    grf_oracle_philox(ctr, key, x);
                    k = (int32_t)(((uint64_t)x[2 * (step & 1) + 1] * (uint64_t)(uint32_t)deg) >> 32);
                }
                const double wgt = data[s + k];
                volatile double scaled = (double)deg * wgt;
                scaled = scaled / one_minus_p;
                if (load_mode == 0) {
                    volatile double nl = load[w] * scaled;
                    load[w] = nl;
                } else if (load_mode == 1) {
                    load[w] = scaled;
                } else {
                    load[w] = wgt;
                }
                cur[w] = indices[s + k];
            }
        }
    }
    free(recs);
    free(cur);
    free(load);
    free(cont);
    free(rank);
    free(count);
    return r;
}
