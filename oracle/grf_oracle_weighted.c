/*
 * Weight-proportional neighbour draws in plain C (TEST INFRASTRUCTURE ONLY -- see oracle/__init__.py): the
 * bit-level answer of grf_alias_records and grf_walk_weighted (definitions at GrfAliasEdge in
 * include/grf_b200.h).
 *
 * Compiled into its own library together with oracle/grf_oracle.c, whose Philox, record sort, result type and
 * accessors (grf_oracle_nnz / _visits / _copy / _free) it reuses unchanged.  The table is built by the
 * sequential sweep of the definition (the device splits it into searches over prefix sums); the walks advance
 * one step at a time per start node, and every length's visits are merged as grf_oracle_build merges them.
 */
#include "grf_oracle.c"

typedef struct {
    double scaled;
    double scaled_alias;
    int32_t col;
    int32_t col_alias;
    uint32_t thr;
    int32_t pad;
} OAliasEdge; /* GrfAliasEdge */

#define T32 4294967296ull

/* S of one row: 32 lane-strided partial sums in index order, then the fixed tree 16, 8, 4, 2, 1 */
double grf_oracle_alias_sum(int32_t d, const double *w) {
    volatile double s[32];
    for (int l = 0; l < 32; ++l) s[l] = 0.0;
    for (int32_t k = 0; k < d; ++k) s[k & 31] = s[k & 31] + fabs(w[k]);
    for (int h = 16; h > 0; h >>= 1)
        for (int l = 0; l < h; ++l) s[l] = s[l] + s[l + h];
    return s[0];
}

/* masses m_k of one row with S > 0, deficit included; returns S */
double grf_oracle_alias_masses(int32_t d, const double *w, uint64_t *m) {
    const double S = grf_oracle_alias_sum(d, w);
    if (!(S > 0.0)) {
        for (int32_t k = 0; k < d; ++k) m[k] = T32;
        return S;
    }
    const double D = (double)d * 4294967296.0;
    uint64_t total = 0;
    int32_t big = 0;
    for (int32_t k = 0; k < d; ++k) {
        volatile double x = fabs(w[k]) * D;
        x = x / S;
        m[k] = (uint64_t)floor(x);
        total += m[k];
        if (m[k] > m[big]) big = k;
    }
    m[big] = (uint64_t)((int64_t)m[big] + ((int64_t)((uint64_t)d * T32) - (int64_t)total));
    return S;
}

/* the records of one row (rs = its first entry) */
static void alias_row(int32_t d, const int32_t *col, const double *w, double one_minus_p, uint64_t *m,
                      int32_t *alias, uint32_t *thr, OAliasEdge *out) {
    const double S = grf_oracle_alias_masses(d, w, m);
    for (int32_t k = 0; k < d; ++k) {
        alias[k] = k;
        thr[k] = 0xffffffffu;
    }
    if (S > 0.0) {
        int32_t li = 0, h = 0;
        while (h < d && m[h] <= T32) ++h;
        if (h < d) {
            while (li < d && m[li] >= T32) ++li;
            int64_t r = (int64_t)m[h];
            for (;;) {
                if (r > (int64_t)T32) {
                    thr[li] = (uint32_t)m[li];
                    alias[li] = h;
                    r -= (int64_t)(T32 - m[li]);
                    ++li;
                    while (li < d && m[li] >= T32) ++li;
                } else {
                    int32_t nh = h + 1;
                    while (nh < d && m[nh] <= T32) ++nh;
                    if (r < (int64_t)T32) {
                        thr[h] = (uint32_t)r;
                        alias[h] = nh;
                        r = (int64_t)m[nh] - (int64_t)(T32 - (uint64_t)r);
                    } else {
                        if (nh >= d) break;
                        r = (int64_t)m[nh];
                    }
                    h = nh;
                }
            }
        }
    }
    volatile double q = S / one_minus_p;
    for (int32_t k = 0; k < d; ++k) {
        const double sk = S > 0.0 ? (w[k] < 0.0 ? -q : q) : 0.0;
        const int32_t a = alias[k];
        const double sa = S > 0.0 ? (w[a] < 0.0 ? -q : q) : 0.0;
        out[k].scaled = sk;
        out[k].scaled_alias = sa;
        out[k].col = col[k];
        out[k].col_alias = col[a];
        out[k].thr = thr[k];
        out[k].pad = 0;
    }
}

int32_t grf_oracle_alias_edge_bytes(void) { return (int32_t)sizeof(OAliasEdge); }

/* records of every row: out [nnz] in the GrfAliasEdge layout */
void grf_oracle_alias_records(int64_t n_nodes, const int32_t *indptr, const int32_t *indices, const double *data,
                              double p_halt, void *out) {
    int32_t dmax = 0;
    for (int64_t v = 0; v < n_nodes; ++v)
        if (indptr[v + 1] - indptr[v] > dmax) dmax = indptr[v + 1] - indptr[v];
    uint64_t *m = (uint64_t *)malloc((size_t)(dmax + 1) * sizeof(uint64_t));
    int32_t *alias = (int32_t *)malloc((size_t)(dmax + 1) * sizeof(int32_t));
    uint32_t *thr = (uint32_t *)malloc((size_t)(dmax + 1) * sizeof(uint32_t));
    OAliasEdge *o = (OAliasEdge *)out;
    for (int64_t v = 0; v < n_nodes; ++v) {
        const int32_t s = indptr[v], d = indptr[v + 1] - s;
        if (d > 0) alias_row(d, indices + s, data + s, 1.0 - p_halt, m, alias, thr, o + s);
    }
    free(m);
    free(alias);
    free(thr);
}

/*
 * Weighted walks: the W walks of a start node advance one step at a time; halting as grf_oracle_build (with
 * `antithetic`, walk 2q+1 halts on walk 2q's halting word XOR 0x80000000); the neighbour from the walk's own
 * neighbour word through the row's alias table; load = load * scaled of the entry taken (cumulative rule).
 */
GrfOracleResult *grf_oracle_build_weighted(int64_t n_nodes, const int32_t *indptr, const int32_t *indices,
                                           const double *data, int64_t start_lo, int64_t start_hi, int32_t W,
                                           int32_t L, double p_halt, int32_t antithetic, uint64_t seed,
                                           int32_t scale_mode) {
    const int64_t nnz = indptr[n_nodes];
    OAliasEdge *tab = (OAliasEdge *)malloc((size_t)(nnz + 1) * sizeof(OAliasEdge));
    grf_oracle_alias_records(n_nodes, indptr, indices, data, p_halt, tab);

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
            for (int32_t w = 0; w < W; ++w) {
                cont[w] = 0;
                if (cur[w] < 0) continue;
                const int32_t deg = indptr[cur[w] + 1] - indptr[cur[w]];
                if (deg == 0) continue;
                const int32_t src = (antithetic && (w & 1)) ? w - 1 : w;
                const uint64_t gid = (uint64_t)start * (uint64_t)W + (uint64_t)src;
                const uint32_t ctr[4] = {(uint32_t)gid, (uint32_t)(gid >> 32), (uint32_t)(step >> 1), 0u};
                uint32_t x[4];
                grf_oracle_philox(ctr, key, x);
                uint32_t xh = x[2 * (step & 1)];
                if (src != w) xh ^= 0x80000000u;
                cont[w] = (uint64_t)xh >= halt_thr;
            }
            for (int32_t w = 0; w < W; ++w) {
                if (!cont[w]) {
                    cur[w] = -1;
                    continue;
                }
                const int32_t s = indptr[cur[w]];
                const int32_t deg = indptr[cur[w] + 1] - s;
                const uint64_t gid = (uint64_t)start * (uint64_t)W + (uint64_t)w;
                const uint32_t ctr[4] = {(uint32_t)gid, (uint32_t)(gid >> 32), (uint32_t)(step >> 1), 0u};
                uint32_t x[4];
                grf_oracle_philox(ctr, key, x);
                const uint64_t P = (uint64_t)x[2 * (step & 1) + 1] * (uint64_t)(uint32_t)deg;
                const OAliasEdge *b = tab + s + (int32_t)(P >> 32);
                const int take_own = (uint32_t)P < b->thr;
                const double fac = take_own ? b->scaled : b->scaled_alias;
                if (fac == 0.0) { /* S = 0: a dead end */
                    cur[w] = -1;
                    continue;
                }
                volatile double nl = load[w] * fac;
                load[w] = nl;
                cur[w] = take_own ? b->col : b->col_alias;
            }
        }
    }
    free(tab);
    free(recs);
    free(cur);
    free(load);
    free(cont);
    return r;
}
