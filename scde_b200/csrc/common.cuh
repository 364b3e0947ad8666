// common.cuh -- shared declarations for libscde_b200 (sm_100a only).
#pragma once
#include <cuda_runtime.h>
#include <cstdint>
#include <cstdio>

namespace scde {

// Row stride (in doubles) of the log-posterior table and of the joint-posterior matrices on the device.
// The default grid has K = 401 points (R/functions.R:237-239); 416 = 2 x 208 keeps every row 128-byte aligned
// and splits into the two 208-wide halves the tiled contraction kernel works on.
constexpr int KP_TILED = 416;
constexpr int WP_TILED = 104;  // bootstrap columns per pass of the tiled kernel (n.randomizations = 100 -> one pass)
constexpr int WS_TILED = 108;  // row stride of the multiplicity matrix W (104 + 4 pad: bank-conflict-free fragment loads)

inline int round_up(int x, int m) { return (x + m - 1) / m * m; }

// error reporting (api.cu)
void set_error(const char *fmt, ...);
int cuda_fail(cudaError_t e, const char *what, const char *file, int line);

#define SCDE_CUDA(expr)                                                                   \
    do {                                                                                  \
        cudaError_t _e = (expr);                                                          \
        if (_e != cudaSuccess) return ::scde::cuda_fail(_e, #expr, __FILE__, __LINE__);   \
    } while (0)

// ---- lp_table.cu ---------------------------------------------------------------------------------
struct CellPrep {  // per-cell grid vectors, each [n_cells][ld]
    double *mu, *lcfp, *lcfpr, *theta;  // theta only for local-theta models
    double *maxcfp;                     // [n_cells]
    int ld;
    // constant-theta fast path (NULL = use the general saddle-point kernel): drop-out probability and the
    // negative binomial's log p_k = -log1p(mu_k/theta), log q_k = -log1p(theta/mu_k)
    double *cfp, *l1, *l2;
    double *scfp;  // [n_cells] sum over the grid of the drop-out probability (fast path)
};
// models: n_cells x 12 column-major with leading dimension ld_models
cudaError_t launch_cell_prep(const double *models, int ld_models, int n_cells, const double *mag, int K,
                             int local_theta, int sqlogit, CellPrep prep, cudaStream_t st);
// A range of cells processed by one launch of the row-level kernels: cells [c0, c1) of row_off (device), i.e. table rows
// [row_off[c0], min(row_off[c1], row_cap)) -- the bounds are read on the device, so a launch can be queued before the
// host knows them (the chunked front of scde_b200_expression_difference).
struct CellRange {
    int c0, c1;
    int64_t row_cap;
};
// row_cell[r] = cell of table row r (from row_off)
cudaError_t launch_row_cell(const int32_t *row_off, CellRange cr, int32_t *row_cell, cudaStream_t st);
// zero_row[c] = the row of cell c whose count is 0, or -1
cudaError_t launch_zero_rows(const int32_t *row_off, const int32_t *row_x, int n_cells, int32_t *zero_row, int64_t row_cap,
                             cudaStream_t st);
// based[c] = 1 when cell c has a zero-count row and that row holds no "log 0" sentinel (it can be subtracted)
cudaError_t launch_based_flags(const double *table, int ld_table, int K, double sentinel, const int32_t *zero_row,
                               int n_cells, int32_t *based, cudaStream_t st, int zero_compact_c0 = -1);
// zero_compact_c0 >= 0: the FP64 table is the COMPACT one -- one row per cell, its zero-count row, at the cell's index --
// and zero_row / based point at cell zero_compact_c0 (the fused fixed-point path stores no other FP64 row, so the table is
// n_cells rows instead of one per distinct (cell, count): 33 MB instead of 40 GB at config 4)
// One warp per table row.  Writes table[r*ld_table + k] (k >= K zero-filled up to ld_table) and row_mode[r] (first
// argmax, before the clamp).  which: 0 = every row, plain values; 1 = only the zero-count rows (plain values);
// 2 = every row except the zero-count ones, stored as the difference to the cell's zero-count row when based[cell].
cudaError_t launch_lp_rows(const double *models, int ld_models, CellRange cr, const int32_t *row_off,
                           const int32_t *row_cell_map, const int32_t *row_x, CellPrep prep, int K,
                           int local_theta, double sentinel, double *table, int ld_table, int32_t *row_mode, int which,
                           const int32_t *zero_row, const int32_t *based, void *row_const, const int32_t *row_snap,
                           int write_f64, int8_t *qtable, uint32_t *row_range, cudaStream_t st, int legacy_q_rows = 0,
                           unsigned long long *work_counter = nullptr, int zero_compact = 0, int8_t *qbound = nullptr);
// legacy_q_rows: build fixed-point-only rows with the per-element kernel the register-resident one replaced (tests)
// work_counter: one device word the register-resident row kernel hands its row chunks out from (zeroed by the launcher;
// required whenever that kernel is chosen, i.e. qtable != NULL with which == 2 on the constant-theta path)
// zero_compact: `table` is the compact FP64 table (see launch_based_flags); which == 1 writes a cell's zero-count row at the
// cell's index, which == 2 reads it there
// write_f64 = 0: the FP64 row is not stored (table is still read for the zero-count rows); qtable != NULL: also emit the
// row's fixed-point planes and its non-sentinel range (contract_i8.cu) -- both only on the constant-theta fast path -- and,
// when qbound != NULL, its bound row (Q_BW bytes per row)
// per-row constants of the constant-theta fast path (4 doubles per row), one thread per row
// ... and row_snap[r] = grid point where the reference's snap rule replaces mu_k by the count, or -1 (needs prep.mu)
cudaError_t launch_row_consts(const double *models, int ld_models, const int32_t *row_off, CellRange cr,
                              const int32_t *row_cell, const int32_t *row_x, void *row_const, int32_t *row_snap,
                              CellPrep prep, int K, cudaStream_t st);

// ---- dedup.cu ------------------------------------------------------------------------------------
// counts: column-major with leading dimension ld_counts; genes [g0, g0+G) of n_cells columns.
// Pass 1: n_unique[c].  Pass 2 (after an exclusive scan into row_off): row_x[row_off[c] + i] = i-th smallest
// distinct count of cell c; ridx[g*ld_ridx + c] = row id of counts[g0+g, c].  err_flag: 1 = negative count,
// 2 = more distinct values than the hash capacity.
// scratch: dedup_scratch_words(n_cells) uint32 words, written by the count pass and read by the emit pass of the same cells
size_t dedup_scratch_words(int n_cells);
cudaError_t launch_dedup_count(const int32_t *counts, int64_t ld_counts, int g0, int G, int n_cells,
                               int32_t *n_unique, int32_t *err_flag, uint32_t *scratch, cudaStream_t st);
// out[i] = base + sum of in[0..i), out[n] = base + total; base = *base_dev (device) or 0 when NULL
cudaError_t launch_exclusive_scan(const int32_t *in, int32_t *out, int n, const int32_t *base_dev, cudaStream_t st);
cudaError_t launch_dedup_emit(const int32_t *counts, int64_t ld_counts, int g0, int G, int n_cells,
                              const int32_t *row_off, int32_t *row_x, int32_t *ridx, int ld_ridx,
                              int32_t *err_flag, int64_t row_cap /* rows row_x can hold */, const uint32_t *scratch,
                              cudaStream_t st);
// (ucl, uci)-given form: ridx[g*ld_ridx + c] = ucl_off[c] + uci[g + G*c]
cudaError_t launch_uci_to_ridx(const int32_t *uci, int G, int n_cells, const int32_t *ucl_off, int32_t *ridx,
                               int ld_ridx, cudaStream_t st);

// ---- boot_contract.cu ----------------------------------------------------------------------------
// W = multiplicity of each cell among each boot's draws, pass-major: W[b / 104][cell][108] (column b % 104) with n_w_rows
// (>= round_up(n_list, 8)) rows per pass, rows beyond n_list zero.  boot_idx: n_boot x D (draw order).
cudaError_t launch_build_w(const int32_t *boot_idx, int n_boot, int D, int n_list, double *W, int n_w_rows,
                           cudaStream_t st);
// Per-gene entry lists: entry e of gene g is (table row lists.row[g*ld + e], W row lists.cell[g*ld + e]); lists.len[g]
// entries, padded to a multiple of 8 with entries that contribute nothing.  order[] = processing order of the genes.
struct GeneLists {
    int32_t *row, *cell, *len, *order;
    int ld;  // multiple of 8, >= round_up(longest list, 8)
};
// zero_row == NULL: dense lists (every cell of the joint).  Otherwise the zero-base form: only cells whose row differs
// from the cell's zero-count row (or whose cell is not `based`) are listed, and the genes are ordered heaviest first.
cudaError_t launch_build_lists(const int32_t *ridx, int ld_ridx, const int32_t *cell_ids, int n_list, int n_genes,
                               const int32_t *zero_row, const int32_t *based, int pad_row, GeneLists out,
                               unsigned long long *total_entries /* += sum of list lengths, may be NULL */,
                               cudaStream_t st, int hot_rank = -1, int count_times = 1);
// hot_rank >= 0 (tcgen05 kernel only): entries whose table row is at most hot_rank rows above the cell's zero-count row
// -- the cell's smallest counts, rows are in ascending count order -- carry LIST_HOT_BIT in out.cell
// Z[pass*104 + b][k] = sum over based cells of the joint of W[cell][b] * table[zero_row[cell]][k]; scratch holds
// base_sum_scratch_doubles() doubles.  Two deterministic passes (partials per cell chunk, then a fixed-order reduction).
size_t base_sum_scratch_doubles(int n_boot, int ld_table);
cudaError_t launch_base_sum(const double *table, int ld_table, const int32_t *zero_row, const int32_t *based,
                            const int32_t *cell_ids, int n_list, const double *W, int n_w_rows, int n_boot, double *Z,
                            double *scratch, cudaStream_t st, int zero_compact = 0);
struct ContractArgs {
    const double *table;   // [rows][ld_table]
    int ld_table;
    GeneLists lists;
    const double *W;  // pass-major [ceil(n_boot/104)][n_w_rows][108]; rows >= (number of cells) are zero
    int n_w_rows;
    int n_boot;       // columns of W that are real
    const double *Z;  // [ceil(n_boot/104)*104][ld_table] initial value of T, or NULL (dense lists)
    // Draw sets: gene_set[gene] (NULL: one set) selects the W and Z of the gene's set, which start gene_set[gene] *
    // set_w_rows rows of W ([set][pass][n_w_rows][108]) and gene_set[gene] * set_z doubles of Z after the first set's
    const int32_t *gene_set;
    int64_t set_w_rows, set_z;
    double scale;     // jp += softmax / scale   (n_boot for the live path, 1 for the legacy / no-bootstrap forms)
    int n_genes, K;
    double *jp;  // [n_genes][ld_jp], must be zeroed by the caller
    int ld_jp;
    int debug = 0;  // tiled kernel: diagnostic mode (scde_b200_options::debug_contract)
};
cudaError_t launch_contract_generic(const ContractArgs &a, cudaStream_t st, int *n_launches);
// requires K <= 416 and ld_table == 416; t_scratch holds contract_tiled_scratch_doubles(n_genes) doubles (the raw
// T[boot, grid] tiles between the contraction and the soft-max kernel)
size_t contract_tiled_scratch_doubles(int n_genes);
cudaError_t launch_contract_tiled(const ContractArgs &a, int n_sm, double *t_scratch, cudaStream_t st, int *n_launches);
bool contract_tiled_supported(const ContractArgs &a);
// ensemble form (src/jpmatLogBoot.cpp:224-237), all cells of the table
cudaError_t launch_ensemble(const double *table, int ld_table, const int32_t *ridx, int ld_ridx, int n_cells, int n_genes,
                            int K, double *jp, int ld_jp, double *rownorm_scratch, int64_t n_rows, cudaStream_t st);
// gathers for return_individual: modes[g + G*c] = mag[row_mode[ridx]], post[c][g + G*k] = table row (clamped)
cudaError_t launch_gather_modes(const int32_t *ridx, int ld_ridx, int G, int n_cells, const int32_t *row_mode,
                                const double *mag, double *modes, cudaStream_t st);
cudaError_t launch_gather_post(const int32_t *ridx, int ld_ridx, int G, int n_cells, const double *table,
                               int ld_table, int K, double sentinel, double minlogprob, double *post,
                               cudaStream_t st);
cudaError_t launch_transpose_out(const double *src, int ld_src, int G, int K, double *dst, cudaStream_t st);
cudaError_t launch_transpose_in(const double *src, int G, int K, double *dst, int ld_dst, cudaStream_t st);
cudaError_t launch_fp64_peak(double *sink, int iters, int blocks, cudaStream_t st);
// the soft-max over the grid and the average over boots that follows either tiled contraction kernel: T is
// [n_pos][104][416] raw T[boot, grid] of the genes order[0 .. n_pos); jp[gene][k] (+)= sum_b softmax_k(T[b, :]) / scale
cudaError_t launch_softmax_avg(double *T, const int32_t *order, int K, int n_boot_pass, double scale, double *jp,
                               int ld_jp, int accumulate, int n_pos, cudaStream_t st);
int contract_tiled_max_genes();  // genes per launch of a tiled kernel (bounds the T scratch)

// ---- contract_i8.cu ------------------------------------------------------------------------------
// Fixed-point form of the table for the tcgen05 (kind::i8) contraction: value = 2^-Q_FRAC * sum_{p < Q_NV} 256^p d_p with
// signed 8-bit digits d_p.  A row is stored as pieces of Q_PIECE = 512 bytes, one per Q_PW = 102 grid points:
// [piece][plane][102] (+ 2 zero bytes), so that one piece is exactly the 512 accumulator columns of an SM's tensor memory
// and a row of the default grid (K = 401) is 2048 bytes.  The reference's "log 0" sentinel (-DBL_MAX/n/1.1) is not a
// plane: every row carries the range [klo, khi] of its grid points that are NOT the sentinel (they form one interval for
// every row the error models produce; a row where they do not is marked Q_RANGE_IRREGULAR and sends the call to the FP64
// kernel), and a grid point of a (gene, boot) is "log 0" exactly when it lies outside the intersection of the ranges
// of the drawn rows (sentinel_range_kernel).
constexpr int Q_NV = 5;           // value planes
constexpr int Q_FRAC = 29;        // fractional bits (|value| <= 1000 < 2^10 fits 5 digits)
constexpr int Q_PW = 102;         // grid points per piece: Q_NV * Q_PW = 510 of the 512 tensor-memory columns
constexpr int Q_PIECE = 512;      // bytes per piece
constexpr int Q_MAX_K = 4 * Q_PW; // largest grid the kernel takes (T rows are KP_TILED = 416 wide)
constexpr int Q_WB = 128;         // bytes per int8 W row: 104 boots + zero padding = M of the MMA
constexpr uint32_t Q_RANGE_IRREGULAR = 0xFFFFFFFFu;
inline int q_pieces(int K) { return (K + Q_PW - 1) / Q_PW; }
// Bound rows (DESIGN.md 4.3, "Pruned pieces"): next to its planes every fixed-point row has Q_BW bytes of bounds on its value
// x = 2^29 D, in units of 2^-5 nat (x / 2^24), rounded outwards: slot u < Q_UB_N holds ceil(max x / 2^24) over the row's
// non-sentinel points of grid block [16 u, 16 u + 16) (0 when it has none), slot Q_UB_N + c floor(x / 2^24) at the sample
// point Q_LB_STEP c + Q_LB_OFF (0 at a sentinel).  Slot i is stored as two signed radix-256 digits, bytes i and
// Q_BSLOTS + i, so that the contraction over the drawn rows (the tcgen05 kernel with one 128-byte piece) sums them exactly.
constexpr int Q_BW = 128;
constexpr int Q_BSLOTS = Q_BW / 2;
constexpr int Q_UB_PTS = 16, Q_UB_N = KP_TILED / Q_UB_PTS;  // 26 blocks
constexpr int Q_LB_STEP = 12, Q_LB_OFF = 6, Q_LB_N = 35;     // samples 6, 18, .., 414
static_assert(Q_UB_N + Q_LB_N <= Q_BSLOTS && Q_LB_STEP * (Q_LB_N - 1) + Q_LB_OFF < KP_TILED, "bound row layout");
// a row's bound slot as the two digits of its bound row
__host__ __device__ inline void q_bound_store(int8_t *brow, int slot, int v) {
    const int lo = (int)(int8_t)(v & 0xFF);
    brow[slot] = (int8_t)lo;
    brow[Q_BSLOTS + slot] = (int8_t)((v - lo) >> 8);
}
inline int q_row_bytes(int K) { return q_pieces(K) * Q_PIECE; }
#ifdef __CUDACC__
// the bound row of a fixed-point row from its planes (q: [piece][plane][102], generic address) and its non-sentinel range;
// lanes l, l + LW, .. of a group of LW lanes take the slots.  (The register-resident row kernel computes the same values
// from its registers: lp_table.cu.)
__device__ inline long long q_value_at(const int8_t *q, int k) {
    const int pc = k / Q_PW, i = k - pc * Q_PW;
    long long x = 0;
#pragma unroll
    for (int pl = Q_NV - 1; pl >= 0; --pl) x = x * 256 + q[pc * Q_PIECE + pl * Q_PW + i];
    return x;
}
__device__ inline void q_bound_row(const int8_t *q, int K, uint32_t range, int8_t *brow, int l, int LW) {
    int klo = 0, khi = K - 1;
    if (range != Q_RANGE_IRREGULAR) {
        klo = (int)(range & 0xFFFFu);
        khi = (int)(range >> 16);
    }
    for (int u = l; u < Q_UB_N; u += LW) {
        long long m = INT64_MIN;
        for (int k = max(u * Q_UB_PTS, klo); k < (u + 1) * Q_UB_PTS && k <= khi; ++k) m = max(m, q_value_at(q, k));
        // ceil(x / 2^24) by an arithmetic shift
        q_bound_store(brow, u, m == INT64_MIN ? 0 : (int)((m + ((1ll << 24) - 1)) >> 24));
    }
    for (int c = l; c < Q_LB_N; c += LW) {
        const int k = Q_LB_STEP * c + Q_LB_OFF;
        q_bound_store(brow, Q_UB_N + c, k < K ? (int)(q_value_at(q, k) >> 24) : 0);
    }
}
#endif
// planes and ranges of every row of an FP64 table (ld_table >= K); one warp per row
cudaError_t launch_quantize_rows(const double *table, int ld_table, int K, int64_t n_rows, int8_t *qtable,
                                 uint32_t *row_range, int8_t *qbound, cudaStream_t st);
// W8[pass][row][128] = (int8) W[pass][row][0..104); *flag |= 1 if a multiplicity exceeds 127
cudaError_t launch_w_to_i8(const double *W, int n_w_rows, int n_boot, int8_t *W8, int32_t *flag, cudaStream_t st);
// What the sides of a launch share (see I8Side)
struct ContractI8Args {
    const int8_t *qtable;
    int ldq;
    const uint32_t *row_range;  // [rows] klo | khi << 16 (NULL: no row holds a sentinel)
    GeneLists lists;   // ld a multiple of 32, lists padded to a multiple of 32 with zero-W entries
    int n_w_rows;
    int n_boot;        // boots of every side's joint
    // Draw sets: gene_set[gene] (NULL: one set) selects the W8 and Z of the gene's set, gene_set[gene] * set_w8 bytes and
    // gene_set[gene] * set_z doubles after the first set's (W8 [set][pass][n_w_rows][128], Z [set][pass * 104 + b][416])
    const int32_t *gene_set;
    int64_t set_w8, set_z;
    double scale;
    double sentinel;   // the "log 0" value of the FP64 table
    int K;
    int ld_jp;
    int32_t *err;      // device flag, |= 2 if the kernel's watchdog fired, |= 4 if the sentinel ranges need the FP64 kernel
    unsigned long long *dbg;  // optional [3] cycle counters of the epilogue (see contract_i8.cu), or NULL
    int item_order;    // 0: item = (gene, piece), a gene's pieces on neighbouring SMs; 1: piece-major (all SMs walk the same
                       // 512-byte piece of the rows at the same time, so rows shared between genes are L2 hits more often)
    int hot_rank;      // >= 0: list entries carry bit 30 of `cell` when the row's rank within its cell is <= hot_rank; such
                       // rows are loaded with the L2 evict_last policy, the others evict_first.  < 0: no hints
    int cold_evict_first;  // with hot_rank >= 0: 1 = the other rows are loaded evict_first, 0 = without a priority
    int ring_stages;       // 0 / 10: the full 10-stage ring (200 KB in flight per SM); 7 or 8: a shallower one
    const int8_t *qbound;  // the table's bound rows [rows][Q_BW] (launch_prune_items)
    const int32_t *items;  // launch_contract_i8_pass: contract only the live items, items[0 .. *n_live) (launch_prune_items);
    const int32_t *n_live; // NULL = every item
};
// One side of a launch: the boots of one joint in one pass.  A launch of the contraction (and of the bound pass) computes
// one side or two over the same genes and lists; with two, items come in pairs on neighbouring SMs, so the second gather
// of a table row is an L2 hit.  The two sides are two joints over the same cells (their passes alike), or passes ps and
// ps + 1 of one joint.  The sentinel ranges, the soft-max and the Z extrema are launched per side or per joint.
struct I8Side {
    const int8_t *W8;   // the pass's W rows [n_w_rows][128] of the first draw set
    const double *Z;    // the pass's base sums [104][416] of the first draw set, or NULL
    double *T;          // T tiles [n_pos][104][416] of one launch
    uint32_t *SR;       // sentinel ranges [n_pos][128] of one launch
    const double *zb;   // the joint's Z extrema (launch_z_bounds; pruning)
    double *jp;         // the joint's output [n_genes][ld_jp]
    int pass;
};
constexpr int32_t LIST_HOT_BIT = 1 << 30;  // in GeneLists::cell (W row ids are < 65536)
// n_draws: draws per randomization (the plane sums are combined pairwise in 32 bits: 257 * 128 * draws < 2^31)
bool contract_i8_supported(int K, int ld_table, int ld_lst, int n_draws);
size_t contract_i8_range_words(int n_genes);  // uint32 words of the (gene, boot) sentinel-range scratch
// s.SR[n_pos][128] = sentinel range of every (gene, boot) of genes order[g0 .. g0 + n_pos), boots of the side
// (no-op when a.row_range == NULL)
cudaError_t launch_sentinel_ranges(const ContractI8Args &a, int g0, int n_pos, const I8Side &s, cudaStream_t st);
// one launch over the sides s[0 .. n_sides) (1 or 2): genes order[g0 .. g0 + n_pos) (n_pos <= contract_tiled_max_genes()),
// boots [104 pass, 104 pass + 104) of each side's joint; writes 2^29 * T[boot, grid] as exact 64-bit integers (without the
// zero-count base, without sentinels) into each side's T ([n_pos][104][416], contract_tiled_scratch_doubles()) -- follow
// with launch_softmax_i8.  The kernel stores the boots of side 0's pass: a second side with fewer (a ragged last pass)
// relies on its W rows being zero beyond its boots.
cudaError_t launch_contract_i8_pass(const ContractI8Args &a, int g0, int n_pos, const I8Side *s, int n_sides, int n_sm,
                                    cudaStream_t st);
// the rest of the gene: s.jp[gene][k] (+)= sum_b softmax_k(2^-29 T + Z)[k] / a.scale with the sentinel ranges s.SR (what
// launch_sentinel_ranges wrote; required when a.row_range != NULL); part_scratch: softmax_i8_scratch_doubles(n_pos)
size_t softmax_i8_scratch_doubles(int n_pos);
// live (NULL: every piece): the pieces launch_prune_items left live, whose T tiles are the only ones written
cudaError_t launch_softmax_i8(const ContractI8Args &a, int g0, int n_pos, const I8Side &s, double *part_scratch, int n_sm,
                              cudaStream_t st, const uint8_t *live = nullptr);
// ---- pruning (DESIGN.md 4.3): (gene, piece) items whose grid points the soft-max cannot see are not contracted
// zb: prune_zb_doubles() doubles, the Z extrema of every (set, pass, boot) of a joint (its Z, a.n_boot, a.K), once per joint
size_t prune_zb_doubles(int n_sets, int n_boot);
cudaError_t launch_z_bounds(const ContractI8Args &a, const double *Z, int n_sets, double *zb, cudaStream_t st);
// live[pos] = the pieces not proven invisible for every boot of the sides s[0 .. n_sides) (bound_i8_kernel: the sums of
// the drawn rows' bound rows a.qbound, with the sentinel ranges and Z extrema of each side; an item of a two-sided launch
// is contracted for both); items / *n_live = the live items in launch order for launch_contract_i8_pass; stats (or NULL)
// [0] += items, [1] += live items, [2] / [3] += the same weighted by the gene's list length.  live: prune_live_bytes(n_pos)
// bytes, items: n_pos * q_pieces(K) ints.  lb_out [n_pos][104] / ub_out [n_pos][104][4] (tests, or NULL): side 0's bounds.
size_t prune_live_bytes(int n_pos);
cudaError_t launch_prune_items(const ContractI8Args &a, int g0, int n_pos, const I8Side *s, int n_sides, int n_sm, uint8_t *live,
                               int32_t *items, int32_t *n_live, unsigned long long *stats, cudaStream_t st,
                               double *lb_out = nullptr, double *ub_out = nullptr);
// tests: out_host[0..3) = exp_nonpos(-745), (-746), (-747) on the device (synchronous on st's completion of the copy)
cudaError_t launch_exp_probe(double *out_host, cudaStream_t st);
// tests: turns the integer tiles in s.T into FP64 T (a.sentinel outside the ranges s.SR, no zero-count base), in place
cudaError_t launch_finalize_t(const ContractI8Args &a, int n_pos, const I8Side &s, cudaStream_t st);

// ---- ratio_summary.cu ----------------------------------------------------------------------------
struct RatioContrast {  // one contrast of a batched launch: its joints and its outputs (layouts as in RatioArgs)
    const double *p1, *p2;
    int32_t *idx;
    double *z;
    double *post;
};
struct RatioArgs {
    const double *p1, *p2;  // [n_genes][ld] row-major (gene-major) device matrices
    int ld;
    int n_genes, n;       // n grid points per input row; output has 2n-1 lags
    const double *prior;  // [n] or NULL
    const int32_t *zero_index;  // device, 1-based
    int n_zero;
    int32_t *idx;     // [3][n_genes] (lb, mle, ub), 0-based   (column-major n_genes x 3)
    double *z;        // [n_genes]
    double *post;     // optional [n_genes][ld_post] gene-major normalised posterior
    int ld_post;
    double *raw;      // optional [n_genes][ld_post] un-normalised sliding product (matSlideMult)
    // optional device table [n_contrasts]: one launch over (genes x contrasts), each contrast's p1, p2, idx, z and post
    // replacing the ones above (which are then unused); every entry must have the same outputs present
    const RatioContrast *contrasts;
    int n_contrasts;
};
cudaError_t launch_ratio_summary(const RatioArgs &a, cudaStream_t st);
cudaError_t launch_magnitude(const int32_t *counts, int64_t n, int G, const double *corr_b, const double *corr_a,
                             double *out, cudaStream_t st);


// ---- prior.cu (scde.expression.prior / scde.failure.probability) -----------------------------------
int prior_pass1_blocks(int64_t n);
// out[e] = drop-out probability of element e of a G x C matrix; magnitudes from `mag` (G x C) or, when NULL, from counts
cudaError_t launch_failure_probability(const int32_t *counts, const double *mag, int64_t n, int G, const double *models, int C,
                                       int sq, double *out, cudaStream_t st);
cudaError_t launch_prior_pass1(const int32_t *counts, int64_t n, int G, const double *models, int C, int sq, double *v, double *w,
                               double *part /* [prior_pass1_blocks(n)] */, unsigned long long *vmax_key,
                               unsigned long long *n_finite, cudaStream_t st);
cudaError_t launch_select_hist(const double *v, int64_t n, unsigned long long prefix, int shift, unsigned long long *hist,
                               cudaStream_t st);
cudaError_t launch_prior_bins(const double *v, const double *w, int64_t n, double inv_sum, double lo, double xdelta, int nbin,
                              unsigned long long *bins, cudaStream_t st);
double prior_key_to_double(unsigned long long k);

}  // namespace scde
