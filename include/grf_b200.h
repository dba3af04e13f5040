/*
 * grf_b200 -- C ABI of the B200-native Graph-Random-Feature (GRF) hot path.
 *
 * This header is the drop-in boundary (SURVEY.md 8b).  The reference
 * (MatthewZhang473/Efficient-Gaussian-Process-on-Graphs) is pure Python and has
 * no FFI of its own; each entry point below names the reference code whose work
 * it replaces (paths relative to the reference root).  The ctypes binding a
 * maintainer adds on the reference side is shown in INTEGRATION.md.
 *
 * Conventions
 *   - every pointer is a DEVICE pointer unless it says "host";
 *   - the caller owns every buffer; the library allocates nothing persistent;
 *   - every call is asynchronous on `stream` (a cudaStream_t passed as void*);
 *   - return value 0 = OK, negative = error (grf_last_error() has the text);
 *   - no torch types, no C++ types: plain pointers and sizes.
 *
 * Data layout in HBM
 *   walk graph      CSR: row_ptr int32[N+1], col_idx int32[nnz], val double[nnz]
 *   staging         row r of this GPU owns stage_*[r*stride .. r*stride+stride),
 *                   stride = 1 + (L-1)*W (worst case); inside it the per-length
 *                   segments follow each other (length 0 first), each sorted by
 *                   column with duplicates merged; row_cnt[r*L + l] = its size
 *   step matrices   (reference layout) one CSR per walk length l, concatenated:
 *                   offsets int64[L*n_rows + 1] step-major, col int32, val double
 *   Phi blocks      (matvec layout) block CSR, row-major over (row, length):
 *                   blk_ptr int32[n_rows*L + 1], entries {int32 length<<27 | col; float val};
 *                   the L segments of a row are contiguous, so blk_ptr[r*L] and
 *                   blk_ptr[(r+1)*L] bound the whole row
 *   Phi^T blocks    same, over (column, length), entries {int32 length<<27 | local_row; float val}
 */
#ifndef GRF_B200_H
#define GRF_B200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define GRF_B200_ABI_VERSION 8

enum {
    GRF_OK = 0,
    GRF_ERR_INVALID = -1,     /* bad argument (the wrapper raises ValueError) */
    GRF_ERR_CUDA = -2,        /* CUDA runtime failure (RuntimeError) */
    GRF_ERR_UNSUPPORTED = -3  /* size outside what this build supports */
};

enum { GRF_DRAW_PHILOX = 0, GRF_DRAW_REPLAY = 1 };
/* Coupled draws of the W walks of one start node (native Philox draws only; OR them into draw_mode).
 * Every walk keeps its marginal law, so every M_l stays unbiased; see GrfWalkCfg.seed for the definitions. */
enum { GRF_DRAW_COUPLE_HALT = 2, GRF_DRAW_COUPLE_NEIGHBOURS = 4 };
/* load rule: sparse_sampler.py:54 & sampler.py:58 | sampler.py:183 | sampler.py:180-181 */
enum { GRF_LOAD_CUMULATIVE = 0, GRF_LOAD_LAST_STEP = 1, GRF_LOAD_ABLATION = 2 };
/* "/ num_walks": scipy csr / W == * (1/W) (sparse_sampler.py:130) | true division (sampler.py:201) */
enum { GRF_SCALE_MUL_RECIP = 0, GRF_SCALE_DIV = 1 };
enum { GRF_ORDER_ROW_MAJOR = 0, GRF_ORDER_STEP_MAJOR = 1 };

/* One stored element of Phi (or Phi^T) in the matvec layout: `col` holds the
 * column (Phi) or local row (Phi^T) in its low GRF_ENTRY_STEP_SHIFT bits and
 * the walk length l of the M_l it belongs to in the bits above, so N and the
 * rows per GPU are limited to 2^27 and L to 32. */
#define GRF_ENTRY_STEP_SHIFT 27
typedef struct {
    int32_t col;
    float val;
} GrfEntry;

/* The walk graph = what SparseRandomWalk.__init__ keeps (sparse_sampler.py:62-70):
 * indptr / indices (int32) and data.astype(float). */
typedef struct {
    int64_t n_nodes;
    int64_t nnz;
    const int32_t *row_ptr;
    const int32_t *col_idx;
    const double *val;
} GrfGraph;

/* One edge of the walk graph as the walker reads it: the neighbour and the load factor
 * (deg(row) * val) / (1 - p_halt) of sparse_sampler.py:54 side by side, so that a step costs one
 * 16-byte gather instead of two from separate arrays (grf_edge_records builds them once per graph
 * and p_halt; on graphs that miss L2 every gathered sector is DRAM traffic). */
typedef struct {
    double scaled;
    int32_t col;
    int32_t pad;
} GrfEdge;

/* Weight-proportional neighbour draws (grf_walk_weighted): one bucket of a row's alias table, 32 bytes = one
 * sector.  Bucket k of a row holds its own entry (col, scaled) and its alias (col_alias, scaled_alias);
 * scaled = sign(w) * S / (1 - p_halt) of that entry, the load factor of a step through it.
 *
 * Definition, for row i with d entries, weights w_k and a_k = |w_k| (k = 0 .. d-1, CSR order):
 *   S       float64: s_l = sum of a_k over k = l, l + 32, l + 64, ... in that order from 0.0 (l = 0 .. 31),
 *           then for h = 16, 8, 4, 2, 1: s_l = s_l + s_{l+h} (l < h); S = s_0.
 *   masses  m_k = (uint64)floor((a_k * D) / S), D = d * 2^32, float64 multiply then divide, no contraction.
 *           The deficit d * 2^32 - sum m_k (int64, may be negative) is added to the largest m_k (lowest index
 *           among ties).  Rows whose |w| are all equal get m_k = 2^32 exactly.
 *   table   T = 2^32.  Light items (m < T) and heavy items (m > T) are each taken in index order (Vose's
 *           method, sweeping form of Huebschle-Schneider & Sanders 2019): h = first heavy, r = m_h; loop:
 *             r > T:  the next light item k gets thr_k = m_k, alias_k = h; r -= T - m_k
 *             r < T:  bucket h gets thr_h = r, alias_h = h' = the next heavy item; r = m_h' - (T - r); h = h'
 *             r = T:  bucket h is full; h = the next heavy item (none: done), r = m_h.
 *           A full bucket (m_k = T, or a heavy item left at exactly T) has thr = 0xffffffff and aliases
 *           itself.  Everything after the masses is integer arithmetic: one exact table per row.
 *   S = 0   (only explicit zeros): every bucket is full with scaled = 0.0, the walk stops there (a dead end).
 *   draw    with the neighbour word x of the Philox schedule of GrfWalkCfg.seed (same counter, same word):
 *           P = (uint64)x * d, j = P >> 32 (the uniform draw's index), frac = (uint32)P; the walk takes
 *           bucket j's entry if frac < thr_j, else its alias.  Entry k is taken with probability m_k / 2^32 / d,
 *           |w_k| / S up to d / 2^32; w = 0 is never taken.  load = load * scaled of the entry taken.
 * On a row whose weights are all +-1 every bucket is full and the draw is the uniform one; the factor
 * sign(w) * (d / (1 - p)) equals (d * w) / (1 - p): the weighted walk is then bit-identical to grf_walk. */
typedef struct {
    double scaled;
    double scaled_alias;
    int32_t col;
    int32_t col_alias;
    uint32_t thr;
    int32_t pad;
} GrfAliasEdge;

/* Arguments of _worker_walks (sparse_sampler.py:26-31) plus the shard and the
 * draw source. */
typedef struct {
    int64_t start_lo, start_hi; /* this GPU's start nodes = its rows of every M_l */
    int32_t walks_per_node;     /* W */
    int32_t max_walk_length;    /* L */
    double p_halt;
    int32_t draw_mode;          /* GRF_DRAW_PHILOX | GRF_DRAW_COUPLE_* flags, or GRF_DRAW_REPLAY alone */
    int32_t load_mode;          /* GRF_LOAD_* */
    uint64_t seed;              /* Philox key (native mode): counter (walk_lo, walk_hi, step/2, 0); words
                                 * (0,1) of the block halt / pick at the even step, (2,3) at the odd one;
                                 * halt iff word < floor(p_halt * 2^32); neighbour = (word * deg) >> 32.
                                 * A dead end (deg = 0) stops a walk without a draw.
                                 * GRF_DRAW_COUPLE_HALT (antithetic termination): walks pair up as
                                 *   (2q, 2q+1), 2q+1 < W (an odd W leaves the last walk unpaired); walk
                                 *   2q+1 halts on the halting word of walk 2q (same step, taken from its
                                 *   counter whether or not walk 2q is still alive) XOR 0x80000000.
                                 *   Neighbour words are unchanged.
                                 * GRF_DRAW_COUPLE_NEIGHBOURS (repelling neighbours): at step s, the
                                 *   m walks of one start node that stand on node v, are still walking
                                 *   and do not halt at s, taken in walk order (rank j), share the group
                                 *   word U = word 0 of philox(counter = (start, v, s, 1)):
                                 *   c = (U * deg(v)) >> 32, and rank j takes neighbour index
                                 *   (c + floor(j * deg(v) / m)) mod deg(v) (64-bit integers); its own
                                 *   neighbour word is unused.  m <= deg: m distinct neighbours; m > deg:
                                 *   floor(m/deg) or ceil(m/deg) walks per neighbour.
                                 * Visits of one (start, length, node) are summed in walk order into a
                                 * double that starts at 0.0 in every mode. */
    /* replay mode: the reference's PCG64 draws, [walk_id*L + step], walk_id =
     * start*W + w; trace_u = rng.random() (NaN where none was drawn), trace_k =
     * rng.integers(deg) (-1 where none) -- sparse_sampler.py:47,51 */
    const double *trace_u;
    const int32_t *trace_k;
    /* optional: edge records from grf_edge_records for this p_halt (NULL: col_idx / val are gathered
     * separately and the factor is computed per step, same roundings) */
    const GrfEdge *edges;
    /* optional (device int32 [n_nodes][L], zeroed by the caller before the first launch of a shard):
     * += 1 per emitted entry at (column, length) -- the segment sizes of the Phi^T blocks, so that
     * grf_transpose_offsets need not re-read the entries to count them */
    int32_t *col_counts;
    /* replay mode: walk id of element 0 of trace_u / trace_k (0 = the trace covers the whole graph; a
     * trace recorded for a row slice starts at start_node * W) */
    int64_t trace_walk_base;
    /* optional output mode for the matvec layout: merged records leave the walker as finished Phi
     * entries {length << 27 | col, (float)(sum "/ W")} in stage_entries [n_local * stage_stride]
     * (same slots as stage_col / stage_sum, which may then be NULL); scale_mode as grf_compact_blocks */
    GrfEntry *stage_entries;
    int32_t scale_mode;
} GrfWalkCfg;

/* Optional split of long rows (hub columns of a power-law Phi^T hold 10^5..10^6 entries): rows
 * with more than `threshold` entries are cut into chunks that are multiplied by separate
 * thread groups into `partial` and then summed per row in chunk order (deterministic). */
typedef struct {
    int32_t threshold;
    int32_t n_long;
    int32_t n_chunks;
    const int32_t *rows;         /* [n_long] ids of the long rows (device) */
    const int32_t *chunk_ptr;    /* [n_long + 1] first chunk of each long row (device) */
    const int32_t *chunk_bounds; /* [n_chunks][2] entry range {begin, end} of each chunk (device) */
    float *partial;              /* [n_chunks][ld] workspace (device) */
    int64_t ld;                  /* >= t */
    /* optional (NULL = ascending chunk id): the order in which the chunks are handed to the warps, a
     * permutation of 0 .. n_chunks-1 (device).  Chunks of hub columns of Phi^T are issued by the first
     * local row they gather, so that the chunks in flight at any moment read one sliding window of V that
     * stays in L2 (V itself is larger than L2 at 4 M nodes); results do not depend on the order */
    const int32_t *chunk_order;
} GrfLongRows;

typedef struct {
    int64_t n_rows;  /* local rows (start nodes owned by this GPU) */
    int64_t n_cols;  /* N */
    int64_t row_lo;  /* global index of local row 0 */
    int32_t n_steps; /* L */
    const int32_t *blk_ptr;   /* [n_rows*L + 1] */
    const GrfEntry *entries;  /* col = global column */
    const int32_t *tblk_ptr;  /* [n_cols*L + 1] */
    const GrfEntry *tentries; /* col = LOCAL row */
    /* optional (NULL / 0 = absent): column window {min, max} of every 32 consecutive rows of
     * Phi (win) and of Phi^T (twin), from grf_block_windows; with them a banded Phi is
     * multiplied through a shared-memory tile of the right-hand side */
    const int32_t *win;  /* [ceil(n_rows/32)][2] */
    const int32_t *twin; /* [ceil(n_cols/32)][2] */
    int32_t win_max_width, twin_max_width;
    const GrfLongRows *long_fwd; /* host pointers, NULL = no row of that side is split */
    const GrfLongRows *long_t;
    /* optional: ids of the columns that have at least one entry in this shard (device, ascending);
     * Phi^T V then visits only those and zero-fills the rest of U */
    const int32_t *tcols;
    int64_t n_tcols;
    int64_t nnz; /* stored entries (0 = unknown); picks the lanes-per-row of the few-column kernels */
    /* optional: two device ints, zero when handed over and private to this GrfPhi (the kernels leave
     * them zero again): the second half of a pass's rows is then handed out warp by warp through a
     * ticket counter instead of by a fixed stride, which evens out the finish times of the SMs.
     * Two products of the SAME GrfPhi must then not run concurrently (same rule as long_*->partial). */
    int32_t *sched;
} GrfPhi;

int grf_abi_version(void);
const char *grf_last_error(void); /* host string, thread-local */

/* Replaces utils_sparse/graph_utils.py:5-30: normalized Laplacian D^-1/2 (D - A) D^-1/2 of a canonical
 * CSR adjacency (sorted columns, no duplicates) on the device, bit-identical to the reference's scipy
 * result.  count: deg / dis (double[n]) and the entries per output row; caller scans
 * (grf_scan_counts(n, 1)) and allocates; fill writes the output CSR (sorted columns). */
int grf_laplacian_count(const GrfGraph *adj, double *deg, double *dis, int32_t *out_cnt, void *stream);
int grf_laplacian_fill(const GrfGraph *adj, const double *deg, const double *dis, const int32_t *out_ptr,
                       int32_t *out_col, double *out_val, void *stream);

/* Edge records {(deg * w) / (1 - p_halt), neighbour} with the reference's rounding order
 * (sparse_sampler.py:54): the walker then skips a float64 division and one gather per step. */
int grf_edge_records(const GrfGraph *graph, double p_halt, GrfEdge *edges /* [nnz] */, void *stream);

/* Staging entries per row the walker may write: 1 + (L-1)*W. */
int64_t grf_walk_stage_stride(int32_t walks_per_node, int32_t max_walk_length);

/* Replaces sparse_sampler.py:26-56 (_worker_walks) and the dict merge at
 * :110-114 (dense twin sampler.py:30-61, :148-186): runs W halting walks from
 * every start node in [start_lo, start_hi), applies the load update in
 * registers, and merges equal (length, node) visits of one start node in
 * shared memory -- loads added in walk order into a double, as the reference's
 * defaultdict does.  Writes stage_col / stage_sum (unscaled sums) and row_cnt;
 * *visits_out (device, may be NULL) += number of walk-steps executed.  With a
 * GRF_DRAW_COUPLE_* bit in cfg->draw_mode the W walks of a start node advance
 * one step at a time with coupled draws (same outputs, same summation). */
int grf_walk(const GrfGraph *graph, const GrfWalkCfg *cfg, int64_t stage_stride, int32_t *stage_col,
             double *stage_sum, int32_t *row_cnt, unsigned long long *visits_out, void *stream);

/* Weight-proportional neighbour draws (no reference counterpart; definitions at GrfAliasEdge): the alias
 * tables of every row for this p_halt (csrc/grf_alias.cu), once per graph and p_halt as grf_edge_records.
 * The weights must be finite (the caller checks). */
int grf_alias_records(const GrfGraph *graph, double p_halt, GrfAliasEdge *out /* [nnz] */, void *stream);

/* grf_walk with neighbour k of a row taken with probability |w_k| / S and the load multiplied by
 * sign(w_k) * S / (1 - p_halt): an unbiased M_l whose per-step factor is bounded by S / (1 - p) (on the
 * normalized Laplacian S <= 1 + sqrt(deg)).  Same outputs as grf_walk.  cfg->draw_mode: GRF_DRAW_PHILOX,
 * optionally | GRF_DRAW_COUPLE_HALT; cfg->load_mode: GRF_LOAD_CUMULATIVE; cfg->edges: NULL; `alias` from
 * grf_alias_records for cfg->p_halt (may be NULL only when no step can be taken: L = 1, p_halt = 1 or nnz = 0). */
int grf_walk_weighted(const GrfGraph *graph, const GrfWalkCfg *cfg, const GrfAliasEdge *alias,
                      int64_t stage_stride, int32_t *stage_col, double *stage_sum, int32_t *row_cnt,
                      unsigned long long *visits_out, void *stream);

/* Exclusive prefix sum of row_cnt[n_rows][L] in row-major or step-major order;
 * offsets has n_rows*L + 1 elements (last = total).  out_is_i64 selects
 * int64_t / int32_t output.  workspace: grf_scan_workspace_bytes(n_rows*L) bytes; after the
 * call its first 8 bytes hold the grand total as int64_t (also when the int32 output wrapped). */
int64_t grf_scan_workspace_bytes(int64_t n_items);
int grf_scan_counts(const int32_t *row_cnt, int64_t n_rows, int32_t n_steps, int32_t order, void *offsets,
                    int32_t out_is_i64, void *workspace, void *stream);

/* Replaces sparse_sampler.py:117-130 (COO -> CSR per length, "/ num_walks") and
 * sampler.py:188-203: staging -> L concatenated CSR matrices (step-major). */
int grf_compact_steps(const int32_t *stage_col, const double *stage_sum, const int32_t *row_cnt,
                      const int64_t *offsets_step_major, int64_t n_rows, int32_t n_steps, int64_t stage_stride,
                      int32_t walks_per_node, int32_t scale_mode, int32_t *out_col, double *out_val, void *stream);

/* Replaces graph_preprocessor.py:117-139 (from_scipy_csr: float32 values) for
 * the matvec: staging -> Phi blocks.  val = (float)(sum * (1/W)). */
int grf_compact_blocks(const int32_t *stage_col, const double *stage_sum, const int32_t *row_cnt,
                       const int32_t *blk_ptr, int64_t n_rows, int32_t n_steps, int64_t stage_stride,
                       int32_t walks_per_node, int32_t scale_mode, GrfEntry *entries, void *stream);

/* Staging already holds finished entries (GrfWalkCfg.stage_entries): gather every row's run to its
 * final place. */
int grf_compact_entries(const GrfEntry *stage_entries, const int32_t *blk_ptr, int64_t n_rows, int32_t n_steps,
                        int64_t stage_stride, GrfEntry *entries, void *stream);

/* Same conversion from the reference layout (a list of L CSR matrices in
 * device memory, e.g. loaded from one of the reference's pickle caches). */
int grf_blocks_from_steps(const int64_t *offsets_step_major, const int32_t *col, const double *val,
                          const int32_t *blk_ptr, int64_t n_rows, int32_t n_steps, GrfEntry *entries, void *stream);
int grf_count_from_steps(const int64_t *offsets_step_major, int64_t n_rows, int32_t n_steps, int32_t *row_cnt,
                         void *stream);

/* Row statistics of Phi or Phi^T blocks in one pass over the row pointers (device int32 census[3]):
 * {rows with more than `threshold` entries, chunks of `threshold` entries they split into,
 * non-empty rows}.  Sizes GrfLongRows and decides whether GrfPhi.tcols pays off; part of the
 * one-off preparation that replaces sparse_lo.py:23-25. */
int grf_row_census(const int32_t *blk_ptr, int64_t n_rows, int32_t n_steps, int32_t threshold, int32_t *census,
                   void *stream);

/* The chunk table of GrfLongRows on the device: rows longer than `threshold` entries in chunks of `chunk` (<=
 * threshold) entries; n_long / n_chunks from grf_row_census() when chunk == threshold.  rows [n_long],
 * chunk_ptr [n_long + 1], chunk_bounds [n_chunks][2] and, with entries, first [n_chunks] = the first X row each
 * chunk gathers (sort it to get chunk_order).  ticket: one device uint64 of scratch.  The order of the rows in
 * the table is not deterministic; the products are (a row adds its own chunks in order). */
int grf_long_rows_build(const int32_t *blk_ptr, const GrfEntry *entries, int64_t n_rows, int32_t n_steps,
                        int32_t threshold, int32_t chunk, int32_t n_long, int32_t n_chunks, unsigned long long *ticket,
                        int32_t *rows, int32_t *chunk_ptr, int32_t *bounds, int32_t *first, void *stream);

/* Multi-GPU row of the path (no reference counterpart: its fork pool merges dictionaries on the host,
 * sparse_sampler.py:90-114).  Start nodes are sharded in contiguous blocks, bounds[g] .. bounds[g+1]
 * (device int64 [world + 1], world <= 64).  mask[v] receives bit g iff a start node of shard g reaches
 * node v within `hops` steps of the walk graph, i.e. a superset of the columns shard g's Phi can
 * touch with max_walk_length = hops + 1.  Columns with >= 2 bits are the only rows of Phi^T V the
 * ranks must sum.  scratch: n_nodes words. */
int grf_shard_reach(const GrfGraph *graph, const int64_t *bounds, int32_t world, int32_t hops,
                    unsigned long long *mask, unsigned long long *scratch, void *stream);

/* Ascending ids of the non-empty rows of Phi or Phi^T blocks (GrfPhi.tcols for a row shard that
 * touches few of the N columns), with no host round trip: the caller sizes `ids` from
 * grf_row_census()[2].  flags [n_rows] receives 0/1 per row (also the "touched" vector the ranks
 * sum to find the columns they share), pos [n_rows + 1] and scan_workspace
 * (grf_scan_workspace_bytes(n_rows)) are scratch. */
int grf_nonempty_rows(const int32_t *blk_ptr, int64_t n_rows, int32_t n_steps, int32_t *flags, int32_t *pos,
                      void *scan_workspace, int32_t *ids, void *stream);

/* Replaces sparse_lo.py:23-25 (.t().to_sparse_csr(), redone on every forward in
 * the reference): build Phi^T blocks once, in two calls that share one workspace of
 * grf_transpose_workspace_bytes(n_cols, L, nnz) bytes:
 *   grf_transpose_offsets  segment sizes per (column, length) and their prefix sum tblk_ptr
 *                          [n_cols*L + 1]; with census_host != NULL (pinned host int32[6]) also the
 *                          grf_row_census of Phi ([0..3)) and Phi^T ([3..6)), copied to the host
 *                          behind the scan so that it arrives while grf_transpose_fill still runs
 *   grf_transpose_fill     the entries sorted by (column, length) with a stable LSD radix sort, so
 *                          every segment is ordered by row (the fixed summation order of Phi^T V);
 *                          tentries[k].col = length << 27 | row, rows counted from the first row passed
 * Both take a ROW BLOCK of Phi: blk_ptr points at the block's first row pointer, n_rows is the
 * block's row count, `entries` is the base of the whole entry array and [entry_lo, entry_lo + nnz)
 * the block's entries.  Transposing a large shard block by block (2^19 rows, say) keeps the rows of V
 * that one block's Phi^T gathers inside L2, and bounds the sort workspace (24 bytes per entry). */
int64_t grf_transpose_workspace_bytes(int64_t n_cols, int32_t n_steps, int64_t nnz);
int grf_transpose_offsets(const int32_t *blk_ptr, const GrfEntry *entries, int64_t n_rows, int64_t n_cols,
                          int32_t n_steps, const int32_t *col_counts /* from GrfWalkCfg, or NULL: counted here */,
                          int32_t *tblk_ptr, void *workspace, int32_t census_threshold, int32_t *census_host,
                          void *stream);
int grf_transpose_fill(const int32_t *blk_ptr, const GrfEntry *entries, int64_t n_rows, int64_t n_cols,
                       int32_t n_steps, int64_t entry_lo, int64_t nnz, void *workspace, GrfEntry *tentries,
                       void *stream);

/* Sparse kernel matrix K = Phi_f Phi_f^T (csrc/grf_kernel_matrix.cu).  Replaces
 * graph_kernels_sparse/fast_grf_kernel_general.py:48-55 (Phi = sum_p f_p M_p by scipy additions, then
 * Phi @ Phi.T by scipy's csr_matmat) with the same float64 roundings, zero-drop and entry order, so that the
 * three arrays equal scipy's element for element.  Shapes: Phi_f n_rows x n_cols, K n_rows x n_rows.
 *   grf_kmat_phi_count / _fill   Phi_f from the step matrices (offsets int64[n_steps*n_rows + 1] step-major),
 *                         using steps p < n_f only (n_f = min(len(f), L) <= 128, f float64: device, or host
 *                         with f_on_host = 1): acc = 0.0, acc = acc + f_p * m over the steps that store the
 *                         entry in ascending p (no FMA; stored zeros of M_p take part), stored iff acc != 0
 *                         (NaN is kept).  count: phi_cnt[n_rows]; caller scans (grf_scan_counts(n_rows, 1),
 *                         int64) -> phi_ptr; fill writes sorted int32 columns and float64 values
 *   grf_kmat_transpose_count / _fill   Phi_f^T as CSR over the n_cols columns: a COUNTING transpose with an
 *                         atomic cursor per column (cursor: int64[n_cols] scratch), so the ORDER OF THE ROWS
 *                         INSIDE A COLUMN IS UNSPECIFIED -- the product only needs the k order, and within one
 *                         k every row j occurs once.  count zeroes and fills tcnt[n_cols]; caller scans
 *                         (int64) -> tptr [n_cols + 1]
 *   grf_kmat_row_sizes    size[i] = min(products of row i, n_rows): an upper bound on the j row i touches
 *   grf_kmat_bin          rows [3][n_rows]: the rows of each bin (order not deterministic, results are);
 *                         stats int64[4] = {rows of bin 0, 1, 2, largest size in bin 2}.  Bins: size <= 256
 *                         warp per row, shared-memory hash; <= 2048 CTA per row, shared-memory hash; larger
 *                         CTA per row with its hash in `workspace` (grf_kmat_workspace_bytes(max_size,
 *                         global_ctas) bytes, global_ctas CTAs).  Every table holds next_pow2(2 * size) slots
 *                         for the row's size; a row that touches more j than its size sets *overflow
 *   grf_kmat_count        sizes from grf_kmat_row_sizes: touched[i] = distinct j (scipy's csr_matmat_maxnnz
 *                         per row), stored[i] = j with sum != 0.  The count COMPUTES THE SUMS (zero-drop
 *                         makes the stored count value-dependent); caller scans stored -> kptr (int64)
 *   grf_kmat_fill         sizes = touched (re-binned): writes row i at kptr[i] in scipy's order, DESCENDING by
 *                         (first k that touched j, j), i.e. not sorted by column
 * bin_rows: HOST int64[3] (stats[0..3) read back); max_size: stats[3].  *overflow (device int32) is zeroed by
 * count / fill and set to 1 if any row outgrew its table or (fill) disagrees with kptr. */
int grf_kmat_phi_count(const int64_t *offsets_step_major, const int32_t *col, const double *val, int64_t n_rows,
                       int32_t n_steps, const double *f, int32_t n_f, int32_t f_on_host, int32_t *phi_cnt,
                       void *stream);
int grf_kmat_phi_fill(const int64_t *offsets_step_major, const int32_t *col, const double *val, int64_t n_rows,
                      int32_t n_steps, const double *f, int32_t n_f, int32_t f_on_host, const int64_t *phi_ptr,
                      int32_t *phi_col, double *phi_val, void *stream);
int grf_kmat_transpose_count(const int64_t *phi_ptr, const int32_t *phi_col, int64_t n_rows, int64_t n_cols,
                             int32_t *tcnt, void *stream);
int grf_kmat_transpose_fill(const int64_t *phi_ptr, const int32_t *phi_col, const double *phi_val, int64_t n_rows,
                            int64_t n_cols, const int64_t *tptr, int64_t *cursor, int32_t *trow, double *tval,
                            void *stream);
int grf_kmat_row_sizes(const int64_t *phi_ptr, const int32_t *phi_col, const int64_t *tptr, int64_t n_rows,
                       int32_t *size, void *stream);
int grf_kmat_bin(const int32_t *size, int64_t n_rows, int32_t *rows, int64_t *stats, void *stream);
int64_t grf_kmat_workspace_bytes(int32_t max_size, int32_t global_ctas);
int grf_kmat_count(const int64_t *phi_ptr, const int32_t *phi_col, const double *phi_val, const int64_t *tptr,
                   const int32_t *trow, const double *tval, int64_t n_rows, const int32_t *size, const int32_t *rows,
                   const int64_t *bin_rows, int32_t max_size, int32_t global_ctas, void *workspace,
                   int64_t workspace_bytes, int32_t *touched, int32_t *stored, int32_t *overflow, void *stream);
int grf_kmat_fill(const int64_t *phi_ptr, const int32_t *phi_col, const double *phi_val, const int64_t *tptr,
                  const int32_t *trow, const double *tval, int64_t n_rows, const int32_t *size, const int32_t *rows,
                  const int64_t *bin_rows, int32_t max_size, int32_t global_ctas, void *workspace,
                  int64_t workspace_bytes, const int64_t *kptr, int32_t *kcol, double *kval, int32_t *overflow,
                  void *stream);

/* Replaces the 2L SparseLinearOperator._matmul calls (sparse_lo.py:16-18), the
 * ConstantMul/Sum operators (sparse_grf_kernel.py:59-61) and the row selection
 * (sparse_grf_kernel.py:32-41) of one kernel matvec
 *     out = Phi[x1] (Phi[x2]^T V),   Phi = sum_l f[l] M_l
 * x1 / x2: GLOBAL row ids (int32) or NULL for "all local rows"; ids outside
 * [row_lo, row_lo + n_rows) are not this GPU's and are skipped (their out rows
 * are left untouched).  V [n2][ldv], out [n1][ldo], U workspace [n_cols][ldu]
 * (= Phi[x2]^T V, this GPU's partial sum: the multi-GPU caller all-reduces it
 * between the two halves); vfull workspace [n_rows][ldu], used when x2 != NULL.  Only columns [0, t)
 * of `out` are written; columns [t, ldu) of U and of vfull are scratch (the kernels may compute and
 * store the padding of the column count to a multiple of 4 there; what they hold never reaches `out`).
 * When x2 selects fewer than 1/16 of the local rows (a BO training set), the first half scatters
 * from those rows of Phi with fp32 atomics instead of passing over Phi^T (cost proportional to the
 * selected rows; summation order not fixed).
 * which: 1 = first half only (U), 2 = second half only (out from U), 3 = both;
 * add 4 to force the global-gather kernel even when column windows are present; add 8 when x2
 * holds no repeated ids and vfull was zero-filled once by the caller (the scatter then needs no
 * memset and no atomics); add 16 to ADD the first half's result to U instead of overwriting it (the
 * second and later row blocks of a shard whose Phi^T was built block by block); add 32 to gather the
 * right-hand side with L1::no_allocate loads (a Phi without column locality: every gathered row is a
 * miss, and not parking it in L1 saves the fill pass through the L1 data stage).  When V is not 16-byte friendly (e.g. t = 17) and vfull is given, V is
 * staged there and the product runs on the column count padded to a multiple of 4. */
int grf_phi_matvec(const GrfPhi *phi, const float *f, const int32_t *x1, int64_t n1, const int32_t *x2,
                   int64_t n2, const float *v, int64_t ldv, float *out, int64_t ldo, float *u, int64_t ldu,
                   float *vfull, int32_t t, int32_t which, void *stream);

/* Column windows for the tiled matvec: win[g] = {min col, max col} over rows [32g, 32g+32)
 * ({INT_MAX, -1} if empty); *max_width (device int32) = widest window. */
int grf_block_windows(const int32_t *blk_ptr, const GrfEntry *entries, int64_t n_rows, int32_t n_steps,
                      int32_t *win /* [ceil(n_rows/32)][2] */, int32_t *max_width, void *stream);

/* Union rows (csrc/grf_union.cu): merge the L per-length segments of every row of Phi (or of
 * Phi^T -- pass tblk_ptr / tentries) on their union pattern, once per Phi.  Work is handed out in TASKS
 * built by the caller: task k = entries [task_b[k], task_e[k]) of row task_row[k] -- a whole row, or one chunk
 * of a long row's flat run (hub columns of a power-law Phi^T hold 10^5..10^6 entries and would serialise a
 * warp); tasks are listed row by row, chunks in order, and cover every entry once.
 *   grf_union_rank   mkey[nnz] = (col << 5 | length), mval[nnz] = values, both in (col, length)
 *                    order inside each row; task_cnt[k] = columns whose first merged entry lies in task k
 *   (caller scans task_cnt -> task_u0 [n_tasks + 1] with grf_scan_counts(n_tasks, 1); the union row pointers
 *    are uptr[r] = task_u0[first task of row r])
 *   grf_union_fill   uhdr[nU] = {col, mask of lengths present}; task_v0[k] = merged position of the task's
 *                    first union entry
 * and, per modulator f, grf_union_materialize writes the plain CSR of Phi_f = sum_l f[l] M_l
 * on that pattern, entries_f[nU] = {col, sum_l f[l] * value}; multiply it with
 * grf_phi_matvec using n_steps = 1, blk_ptr = uptr, f = [1]. */
int grf_union_rank(const int32_t *blk_ptr, const GrfEntry *entries, int32_t n_steps, const int32_t *task_row,
                   const int32_t *task_b, const int32_t *task_e, int64_t n_tasks, uint32_t *mkey, float *mval,
                   int32_t *task_cnt, void *stream);
int grf_union_fill(const int32_t *blk_ptr, const uint32_t *mkey, int32_t n_steps, const int32_t *task_row,
                   const int32_t *task_b, const int32_t *task_e, int64_t n_tasks, const int32_t *task_u0,
                   int32_t *uhdr /* [nU][2] */, int32_t *task_v0, void *stream);
int grf_union_materialize(const int32_t *task_u0, const int32_t *task_v0, int64_t n_tasks, const int32_t *uhdr,
                          const float *mval, const float *f, int32_t n_steps, GrfEntry *entries_f, void *stream);

/* Line-pair layout of the merged Phi_f / Phi_f^T for t = 16 (csrc/grf_pairs.cu): union entries of one row whose
 * columns 2p and 2p+1 share a 128-byte line of X become ONE entry {p, w_even, w_odd, 0} (16 bytes), gathered with
 * one L1 wavefront by 8 lanes.  Pays on lattices, rings and any numbering with locality; the caller compares
 * n_pairs with n_union and keeps grf_phi_matvec otherwise.  Same role as grf_phi_matvec for the CG steady state
 * (sparse_lo.py:16-18 x 2L), whole halves only:
 *   grf_pairs_count  pcnt[r] = pair entries of union row r (uent: the union headers or the merged entries --
 *                    only the column field is read); caller scans -> pptr [n_rows + 1]
 *   grf_pairs_index  pidx[u] = pair slot of union entry u            (both once per Phi)
 *   grf_pairs_fill   pent[n_pairs][4] from the merged entries of one modulator value
 *   grf_pairs_spmm   y[k, 0:16] = sum_{pairs of row k} w_even * x[2p, :] + w_odd * x[2p+1, :]; x [n_x][16] with
 *                    leading dimension 16 and 128-byte alignment; row_ids (or NULL) as in grf_phi_matvec */
int grf_pairs_count(const int32_t *uptr, const GrfEntry *uent, int64_t n_rows, int32_t *pcnt, void *stream);
int grf_pairs_index(const int32_t *uptr, const GrfEntry *uent, int64_t n_rows, const int32_t *pptr, int32_t *pidx,
                    void *stream);
int grf_pairs_fill(const GrfEntry *uent, const int32_t *pidx, int64_t n_union, int64_t n_pairs, int32_t *pent,
                   void *stream);
int grf_pairs_spmm(const int32_t *pptr, const int32_t *pent, const int32_t *row_ids, int64_t n_tasks, int64_t row_lo,
                   int64_t n_rows, const float *x, int64_t n_x, float *y, int64_t ldy, void *stream);

/* both halves on pair entries in one call: which & 1: u = Phi_f^T v (tpptr / tpent: the transposed side, n_cols
 * rows, v [n_rows][16]);  which & 2: out = Phi_f[x1] u (u [n_cols][16]) */
int grf_pairs_matvec(const int32_t *tpptr, const int32_t *tpent, const int32_t *pptr, const int32_t *pent,
                     const int32_t *x1, int64_t n1, int64_t row_lo, int64_t n_rows, int64_t n_cols, const float *v,
                     float *u, float *out, int64_t ldo, int32_t which, void *stream);

/* Per-length reduction for the modulator gradient (what upstream
 * _bilinear_derivative yields for sparse_grf_kernel.py:51-62):
 *   grad[l] += sum_k sum_t left[k][t] * (M_l[x[k], :] @ P)[t]
 * P [n_cols][ldp].  Call twice (left with P = Phi[x2]^T right, right with
 * P = Phi[x1]^T left) for the full derivative.  grad: float[L], accumulated. */
int grf_phi_fgrad(const GrfPhi *phi, const int32_t *x, int64_t n, const float *left, int64_t ldl, const float *p,
                  int64_t ldp, int32_t t, float *grad, void *stream);

/* Replaces the diag=True branch of sparse_grf_kernel.py:55-57 (which multiplies two densified row sets):
 *   dots[i][l] = sum over the length-l entries e of Phi row x1[i] of  e.val * Phi_f[x2[i], col(e)],
 * Phi_f = sum_l f[l] M_l, so that diag(K[x1, x2])[i] = sum_l f[l] * dots[i][l]; the columns of dots are what
 * the modulator gradient of that diagonal needs.  x1 / x2: global row ids (NULL = row i of this shard; then
 * n = n_rows); pairs with a row outside this shard are written as zeros.  dots: float [n][L]. */
int grf_phi_row_dots(const GrfPhi *phi, const float *f, const int32_t *x1, const int32_t *x2, int64_t n,
                     float *dots, void *stream);

/* Exact GP posterior variance at test rows (csrc/grf_posterior.cu; no reference counterpart: its users estimate
 * the variance from SparseGraphGP.predict samples).  With w_e = f[length(e)] * e.val:
 *   q[i] = sum_{c < r} ( sum_{e in row x[i], col_slot[col(e)] >= 0} w_e * C[col_slot[col(e)] * ldc + c] )^2
 *   d[i] = sum_{e in row x[i]} w_e^2                                   (d may be NULL)
 * col_slot int32[n_cols]: the row of C that holds column c of Phi_f, or -1; C [m][ldc] float32 (columns
 * [r, ldc) are never read into a result).  On the merged Phi_f with C = G L^-T of the training rows, d - q is
 * the posterior variance (grf_b200/posterior.py).  x: global row ids (NULL = every local row, n = n_rows); ids
 * outside [row_lo, row_lo + n_rows) give q = d = +0.  Only q[0, n) and d[0, n) are written; the summation order
 * is fixed (no atomics), so repeated calls agree bit for bit. */
int grf_phi_row_quadform(const GrfPhi *phi, const float *f, const int32_t *x, int64_t n, const int32_t *col_slot,
                         const float *C, int64_t ldc, int32_t r, float *q, float *d, void *stream);

/* Row projection onto the training column set (csrc/grf_posterior.cu): with w_e = f[length(e)] * e.val,
 *   out[i * ldo + c] = sum_{e in row x[i], col_slot[col(e)] >= 0} w_e * B[col_slot[col(e)] * ldb + c]    (c < r)
 * col_slot as for grf_phi_row_quadform; B [m][ldb] float32.  With the slot map and factor of
 * grf_b200/posterior.py this is the exact posterior mean (B = G K^-1 y, r = 1), the cross term of the joint
 * covariance (B = C = G L^-T, r = n) and the correction of pathwise samples (B = G K^-1 V, r = samples).
 * x: global row ids (NULL = every local row, n = n_rows); ids outside [row_lo, row_lo + n_rows) give a row of +0.
 * Only columns [0, r) of out are written, and columns [r, ldb) of B never reach a result.  The summation order
 * is fixed (no atomics), so repeated calls agree bit for bit.  Per-length and merged blocks, L <= 32. */
int grf_phi_row_project(const GrfPhi *phi, const float *f, const int32_t *x, int64_t n, const int32_t *col_slot,
                        const float *B, int64_t ldb, int32_t r, float *out, int64_t ldo, void *stream);

/* Rank-k update of the posterior variance (and mean) at fixed test rows after the training set grew
 * (csrc/grf_posterior.cu; grf_b200/posterior.py, ExactPosterior.condition_on and PosteriorMarginals).  With
 * w_e = f[length(e)] * e.val and p_c(i) = sum_{e in row x[i], col_slot[col(e)] >= 0} w_e * B[col_slot[col(e)] * ldb + c]:
 *   q[i]   += sum_{c < r} p_c(i)^2        (the squares in float64, added to q[i] in the order c = 0, 1, ..)
 *   var[i]  = (float)(d[i] - q[i]) with the updated q, clamped at +0 (NaN stays NaN, as torch.clamp_min)
 *   mean[i] = p_r(i)                      (only with with_mean = 1; mean may be NULL when with_mean = 0)
 * k = r + with_mean columns of B [m][ldb] float32 are read, 1 <= k <= 64 and ldb >= k; columns [k, ldb) never
 * reach a result.  B = [C_new | a]: the columns C gained and the new a = G K^-1 y.  q double[n], d float[n] (the
 * prior variance, from grf_phi_row_quadform), var and mean float[n].  col_slot, x and the row shard as for
 * grf_phi_row_project: ids outside [row_lo, row_lo + n_rows) have p = 0, so q stays as it is, var is still written
 * from d and q and mean is +0.  Only elements [0, n) are written; the summation order is fixed (no atomics), so
 * repeated calls agree bit for bit.  k <= 4 runs row_condition_narrow_kernel, k <= 64 row_condition_mid_kernel (the
 * warp shapes of the projection).  -1 for k outside [1, 64], ldb < k, a NULL required pointer, or x NULL with
 * n != n_rows. */
int grf_phi_row_condition(const GrfPhi *phi, const float *f, const int32_t *x, int64_t n, const int32_t *col_slot,
                          const float *B, int64_t ldb, int32_t r, int32_t with_mean, double *q, const float *d,
                          float *var, float *mean, void *stream);

/* Rank-k downdate of the posterior variance (and the mean) at fixed test rows after training rows were removed
 * (csrc/grf_posterior.cu; grf_b200/posterior.py, ExactPosterior.forget and PosteriorMarginals).  The arguments and
 * rules of grf_phi_row_condition, with the squares subtracted:
 *   q[i]   -= sum_{c < r} p_c(i)^2        (the squares in float64, subtracted from q[i] in the order c = 0, 1, ..)
 *   var[i]  = (float)(d[i] - q[i]) with the updated q, clamped at +0 (NaN stays NaN)
 *   mean[i] = p_r(i)                      (only with with_mean = 1)
 * B = [U | a]: U = C Z R^-1 with Z = L^-1 E_B and Z^T Z = R^T R for the removed positions B, so that C C^T - U U^T is
 * the C C^T of the remaining rows, and the new a.  p is summed in exactly the order of grf_phi_row_condition.  k <= 4
 * runs row_downdate_narrow_kernel, k <= 64 row_downdate_mid_kernel.  -1 in the cases of grf_phi_row_condition. */
int grf_phi_row_downdate(const GrfPhi *phi, const float *f, const int32_t *x, int64_t n, const int32_t *col_slot,
                         const float *B, int64_t ldb, int32_t r, int32_t with_mean, double *q, const float *d,
                         float *var, float *mean, void *stream);

/* Per-length Gram of the training rows, light part (csrc/grf_gram.cu; no reference counterpart: the reference
 * estimates the marginal likelihood by CG and probes).  With A[R, c] = M_l[x_i, c] for the E row R = l * n + i,
 * E = A A^T is float64 [n_rows][lde], n_rows = L * n.  The columns the training rows touch are numbered as slots
 * 0 .. n_slots - 1 by the caller (grf_b200/engine.py, PhiBlocks.training_gram):
 *   row_ptr  int32[n_rows + 1], row_ent: the entries of row R as {slot, val}, ascending slot
 *   slot_ptr int32[n_slots + 1], slot_ent: the entries of slot s as {R', val}, each R' at most once
 *   order    int32[n_rows], the order in which the rows are handed to the warps (NULL = ascending R)
 * For every R and every C >= R this adds sum over the slots s shared by R and C of val(R, s) * val(C, s) into
 * E[R * lde + C], the slots in ascending order, each product exact in float64; no other element is touched (the
 * caller zero-fills E, adds the hub slots' dense part and mirrors).  Fixed order, no atomics: repeated calls agree
 * bit for bit. */
int grf_gram_light(const int32_t *order, int64_t n_rows, const int32_t *row_ptr, const GrfEntry *row_ent,
                   const int32_t *slot_ptr, const GrfEntry *slot_ent, int64_t n_slots, double *E, int64_t lde,
                   void *stream);
/* E[C * lde + R] = E[R * lde + C] for every R < C < n_rows (float64): the upper triangle mirrored, exactly. */
int grf_gram_mirror(double *E, int64_t n_rows, int64_t lde, void *stream);

/* The one exchange of the path (SURVEY.md 8e; no reference counterpart: its matvec runs on one device):
 * U <- sum over the GPUs of the partials U_g = Phi_g[x2]^T V_g between the two halves of a product, as one
 * kernel per rank over NVLink peer memory.  peer_u[g] / peer_flags[g] (HOST arrays of `world` DEVICE pointers)
 * are every rank's U buffer and flag block as mapped into this process (torch symmetric memory, cudaIpc...);
 * all U buffers hold n_floats floats in the same layout, 16-byte aligned; a flag block has
 * grf_exchange_flag_bytes(world) bytes, zero-filled once.  Every rank calls this with the same `epoch`,
 * 1, 2, 3, ... per exchange.  On return (in stream order) this rank's U holds the sum -- added in rank
 * order on every rank, so all copies are bit-identical.  The call must not be made by ranks that share a GPU. */
int64_t grf_exchange_flag_bytes(int32_t world);
int grf_exchange_sum(float *const *peer_u, uint32_t *const *peer_flags, int32_t world, int32_t rank,
                     int64_t n_floats, uint32_t epoch, void *stream);
/* The same sum through the NVSwitch (NVLS): multicast_u = the multicast address of the ranks' U buffers (torch
 * symmetric memory: handle.multicast_ptr).  The switch adds the copies on load (multimem.ld_reduce) and replicates
 * the store (multimem.st): 1/G of U crosses this GPU's links each way instead of (G-1)/G.  Flags as above. */
int grf_exchange_sum_nvls(float *multicast_u, uint32_t *const *peer_flags, int32_t world, int32_t rank,
                          int64_t n_floats, uint32_t epoch, void *stream);

/* Fused vector kernels of batched CG on (K + sigma2 I) X = B (csrc/grf_cg.cu); replace the
 * elementwise / reduction launches of upstream linear_cg as called at
 * models/sparse_grf_model.py:43.  Per iteration, after Kd = grf_phi_matvec(d):
 *   grf_cg_dot        ad = Kd + sigma2 * d (in place); partial[b][c] = block b's share of <d, ad>
 *   grf_cg_update     alpha = rs / <d, ad>; x += alpha d; r -= alpha ad; rr_partial = shares of <r, r>
 *   grf_cg_direction  rs_out = <r, r>; d = r + (rs_out / rs) d
 * partial buffers: grf_cg_num_partials(n, t) rows of t floats.  All matrices n x t row-major. */
int32_t grf_cg_num_partials(int64_t n, int32_t t);
int grf_cg_dot(float *ad, int64_t ldad, const float *d, int64_t ldd, float sigma2, int64_t n, int32_t t,
               float *partial, void *stream);
int grf_cg_update(float *x, int64_t ldx, float *r, int64_t ldr, const float *d, int64_t ldd, const float *ad,
                  int64_t ldad, const float *rs, const float *dad_partial, int64_t n, int32_t t, float eps,
                  float *rr_partial, void *stream);
int grf_cg_direction(float *d, int64_t ldd, const float *r, int64_t ldr, const float *rs, const float *rr_partial,
                     int64_t n, int32_t t, float eps, float *rs_out, void *stream);

#ifdef __cplusplus
}
#endif
#endif /* GRF_B200_H */
