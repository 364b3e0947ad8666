// api.cu -- the C ABI of libscde_b200 (include/scde_b200.h): contexts, device buffers, the orchestration of
// scde.posteriors / scde.expression.difference on the device, and nothing else.  No CPU fallback: every compute
// entry point fails with SCDE_B200_ENODEVICE when there is no CUDA device.
#include "../../include/scde_b200.h"
#include "common.cuh"
#include "hostmath.h"

#include <cfloat>
#include <cmath>
#include <cstdarg>
#include <cstring>
#include <string>
#include <chrono>
#include <exception>
#include <map>
#include <memory>
#include <new>
#include <atomic>
#include <thread>
#include <vector>

namespace scde {

static thread_local std::string g_err;

void set_error(const char *fmt, ...) {
    char buf[1024];
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(buf, sizeof(buf), fmt, ap);
    va_end(ap);
    g_err = buf;
}

int cuda_fail(cudaError_t e, const char *what, const char *file, int line) {
    set_error("CUDA error %d (%s) at %s:%d: %s", (int)e, cudaGetErrorString(e), file, line, what);
    if (e == cudaErrorMemoryAllocation) return SCDE_B200_ENOMEM;
    if (e == cudaErrorNoDevice || e == cudaErrorInsufficientDriver) return SCDE_B200_ENODEVICE;
    return SCDE_B200_ECUDA;
}

template <class T>
struct DBuf {  // grow-only device buffer
    T *p = nullptr;
    size_t cap = 0;
    DBuf() = default;
    DBuf(const DBuf &) = delete;
    DBuf &operator=(const DBuf &) = delete;
    ~DBuf() {
        if (p) cudaFree(p);
    }
    cudaError_t ensure(size_t n) {
        if (n <= cap && p) return cudaSuccess;
        if (p) cudaFree(p);
        p = nullptr;
        cap = 0;
        if (n == 0) n = 1;
        cudaError_t e = cudaMalloc((void **)&p, n * sizeof(T));
        if (e == cudaSuccess) cap = n;
        return e;
    }
};

struct StageTimer {
    std::vector<cudaEvent_t> pool;
    struct Span {
        int stage;
        int e0, e1;
    };
    std::vector<Span> spans;
    size_t used = 0;
    int launches[SCDE_B200_T_COUNT] = {0};
    ~StageTimer() {
        for (auto e : pool) cudaEventDestroy(e);
    }
    void reset() {
        spans.clear();
        used = 0;
        memset(launches, 0, sizeof(launches));
    }
    int get() {
        if (used == pool.size()) {
            cudaEvent_t e;
            if (cudaEventCreate(&e) != cudaSuccess) return -1;
            pool.push_back(e);
        }
        return (int)used++;
    }
    int begin(cudaStream_t st) {
        int i = get();
        if (i >= 0) cudaEventRecord(pool[i], st);
        return i;
    }
    void end(int stage, int e0, cudaStream_t st, int n_launch) {
        int i = get();
        if (i >= 0 && e0 >= 0) {
            cudaEventRecord(pool[i], st);
            spans.push_back({stage, e0, i});
        }
        launches[stage] += n_launch;
    }
    void collect(scde_b200_stats *s) {
        for (int i = 0; i < SCDE_B200_T_COUNT; ++i) {
            s->ms[i] = 0;
            s->launches[i] = launches[i];
        }
        for (auto &sp : spans) {
            float ms = 0;
            if (cudaEventElapsedTime(&ms, pool[sp.e0], pool[sp.e1]) == cudaSuccess) s->ms[sp.stage] += ms;
        }
        int tot = 0;
        for (int i = 0; i < SCDE_B200_T_TOTAL; ++i) tot += launches[i];
        s->launches[SCDE_B200_T_TOTAL] = tot;
    }
};

}  // namespace scde

using namespace scde;

namespace {
struct DiffWorkspace;
}

static scde_b200_options default_options() {
    scde_b200_options o;
    memset(&o, 0, sizeof(o));
    o.contract_kernel = 0;
    o.zero_base = 1;
    o.fused_fixed_point = 1;
    o.lp_rows_kernel = 0;
    o.count_chunks = 8;
    o.split_front = 1;
    o.uniform_chunks = 0;
    o.pipeline_front = 1;
    o.item_order = 1;  // piece-major: measured 5 % faster at config 4 (profiles/r02a_sweep.txt)
    o.hot_rank = -1;
    o.cold_evict_first = 1;
    o.twin_batch_joints = 1;
    o.prune_pieces = 1;
    return o;
}

struct scde_b200_ctx {
    int device = 0;
    cudaStream_t stream = nullptr;
    int n_sm = 148;
    scde_b200_options opt = default_options();
    std::vector<scde_b200_ctx *> children;      // scde_b200_create_multi: the contexts of the other devices of the list
    DiffWorkspace *ws = nullptr;  // large device buffers of the differential-expression path, kept across calls
    bool ws_busy = false;
    DBuf<unsigned long long> epi_dbg;       // SCDE_B200_EPI_TIMING: cycle counters of the tcgen05 kernel's epilogue
    cudaStream_t copy_stream = nullptr;     // H2D of the count matrix in cell chunks, overlapped with the table build
    std::vector<cudaEvent_t> copy_events;   // one per chunk (+ 1: "the compute stream has released the counts buffer")
    int32_t *h_draws = nullptr;             // mapped pinned staging of the bootstrap draws of the one-shot call: the W build
    size_t h_draws_cap = 0;                 // reads them in place, so they never queue behind the count copies
};

namespace {

inline int table_ld(int K) { return K <= KP_TILED ? KP_TILED : round_up(K, 8); }

struct LpTable {
    int n_cells = 0, n_genes = 0, K = 0, ld = 0, ld_ridx = 0;
    int64_t n_rows = 0;
    double sentinel = 0;
    DBuf<int32_t> row_off, row_x, row_mode, row_cell, row_snap, ridx, n_unique, err, zero_row, based;
    DBuf<double> table, mu, lcfp, lcfpr, theta, maxcfp, cfp, l1, l2, rowc, scfp;
    DBuf<int8_t> q;      // fixed-point planes of the table (contract_i8.cu), [n_rows][q_row_bytes(K)]
    DBuf<uint32_t> qrange;  // [n_rows] non-sentinel range of every row (klo | khi << 16)
    DBuf<int8_t> qb;        // [n_rows][Q_BW] bound rows of the fixed-point table (pruned contraction)
    DBuf<uint32_t> dedup_bits;  // per-cell bitmaps between the two dedup passes
    DBuf<unsigned long long> work_counter;  // chunk counter of the fixed-point row kernel
    bool want_q = false, has_q = false;
    bool want_bounds = false;  // bound rows whatever the size (scde_b200_probe_table_bounds)
    bool has_bounds = false;   // t.qb holds the bound rows of the fixed-point table
    bool f64_rows = true;  // false: the FP64 rows of non-zero counts were not stored (planes only)
    bool want_modes = true;  // row_mode (argmax of every row) is needed: only for return.individual.posterior.modes
    bool fast_theta = false;  // every corr.theta finite and > 0, no local-theta fit: constant-theta fast path
    // zero-base form: rows of non-zero counts hold lp(x) - lp(0) of their cell, the zero-count rows lp(0) itself, and
    // the contraction only visits the cells whose count is non-zero (boot_contract.cu)
    bool zero_base = false;
    // the FP64 table holds one row per CELL (its zero-count row, at the cell's index) instead of one per table row: set by
    // reserve_rows when the fixed-point planes come from the row kernel itself, which stores no other FP64 row
    bool zero_compact = false;
};

#define TRY(x)                          \
    do {                                \
        int _r = (x);                   \
        if (_r != SCDE_B200_OK) return _r; \
    } while (0)

#define CHECK_CTX(ctx)                                                  \
    do {                                                                \
        if (!(ctx)) {                                                   \
            set_error("null context");                                  \
            return SCDE_B200_EINVAL;                                    \
        }                                                               \
        SCDE_CUDA(cudaSetDevice((ctx)->device));                        \
    } while (0)

// What fill_table decides once per table and the row-level launches need: which kernels, which outputs.
// Pruning (DESIGN.md 4.3) pays where a joint has at least this many cells: measured on one B200 (1000 W), config 3 (1000
// cells per joint) was 3.0 ms per step slower with it (bound pass and bound rows cost more than the 27 % of the gather they
// removed), config 4 (5000) 7.7 ms faster.  The bound rows are only written for tables of at least as many cells.
constexpr int PRUNE_MIN_CELLS = 2500;

struct TablePlan {
    bool fast = false;     // constant-theta fast row kernel
    bool q_any = false;    // the table also exists in fixed point (tcgen05 contraction)
    bool q_fused = false;  // ... emitted by the row kernel itself; the FP64 rows of non-zero counts are then not stored
    CellPrep prep{};
    void *rowc = nullptr;
    int32_t *rmode = nullptr;
    int8_t *qf = nullptr;
    uint32_t *qr = nullptr;
    int8_t *qb = nullptr;
    bool bounds = false;   // the table also gets its bound rows
};

TablePlan plan_table(const scde_b200_ctx *ctx, const LpTable &t, int local_theta) {
    TablePlan pl;
    pl.fast = t.fast_theta && !local_theta && t.K <= KP_TILED;
    pl.q_any = t.want_q && t.zero_base && t.ld == KP_TILED && t.K <= Q_MAX_K;
    pl.q_fused = pl.q_any && pl.fast && ctx->opt.fused_fixed_point;
    pl.bounds = pl.q_any && (t.want_bounds || (ctx->opt.prune_pieces && t.n_cells >= PRUNE_MIN_CELLS));
    return pl;
}

// per-cell buffers (independent of the number of table rows) + the per-cell grid vectors
int prepare_cells(scde_b200_ctx *ctx, LpTable &t, TablePlan &pl, const double *models_dev, int ld_models,
                  const double *mag_dev, int local_theta, int sqlogit) {
    cudaStream_t st = ctx->stream;
    const size_t cl = (size_t)t.n_cells * t.ld;
    SCDE_CUDA(t.mu.ensure(cl));
    SCDE_CUDA(t.lcfp.ensure(cl));
    SCDE_CUDA(t.lcfpr.ensure(cl));
    if (local_theta) SCDE_CUDA(t.theta.ensure(cl));
    SCDE_CUDA(t.maxcfp.ensure(t.n_cells));
    if (pl.fast) {
        SCDE_CUDA(t.cfp.ensure(cl));
        SCDE_CUDA(t.l1.ensure(cl));
        SCDE_CUDA(t.l2.ensure(cl));
        SCDE_CUDA(t.scfp.ensure((size_t)t.n_cells));
    }
    if (t.zero_base) {
        SCDE_CUDA(t.zero_row.ensure((size_t)t.n_cells));
        SCDE_CUDA(t.based.ensure((size_t)t.n_cells));
    }
    pl.prep = CellPrep{t.mu.p, t.lcfp.p, t.lcfpr.p, local_theta ? t.theta.p : nullptr, t.maxcfp.p, t.ld,
                       pl.fast ? t.cfp.p : nullptr, pl.fast ? t.l1.p : nullptr, pl.fast ? t.l2.p : nullptr,
                       pl.fast ? t.scfp.p : nullptr};
    SCDE_CUDA(launch_cell_prep(models_dev, ld_models, t.n_cells, mag_dev, t.K, local_theta, sqlogit, pl.prep, st));
    return SCDE_B200_OK;
}

// per-row buffers for `rows` table rows
int reserve_rows(LpTable &t, TablePlan &pl, size_t rows) {
    t.zero_compact = pl.q_fused && t.zero_base;  // 33 MB instead of 40 GB at config 4
    SCDE_CUDA(t.table.ensure((t.zero_compact ? (size_t)t.n_cells : rows) * t.ld));
    SCDE_CUDA(t.row_mode.ensure(rows));
    SCDE_CUDA(t.row_cell.ensure(rows));
    if (pl.fast) {
        SCDE_CUDA(t.rowc.ensure(4 * rows));
        SCDE_CUDA(t.row_snap.ensure(rows));
    }
    if (pl.q_any) {
        SCDE_CUDA(t.q.ensure(rows * q_row_bytes(t.K)));
        SCDE_CUDA(t.qrange.ensure(rows));
        if (pl.bounds) SCDE_CUDA(t.qb.ensure(rows * Q_BW));
        SCDE_CUDA(t.work_counter.ensure(1));
    }
    pl.rowc = pl.fast ? (void *)t.rowc.p : nullptr;
    pl.rmode = t.want_modes ? t.row_mode.p : nullptr;
    pl.qf = pl.q_fused ? t.q.p : nullptr;
    pl.qr = pl.q_fused ? t.qrange.p : nullptr;
    pl.qb = pl.q_fused && pl.bounds ? t.qb.p : nullptr;
    t.has_bounds = pl.bounds;
    return SCDE_B200_OK;
}

// the row-level kernels for the cells of `cr` (their rows are read from t.row_off on the device); returns the number of
// launches through *nl
int launch_table_rows(scde_b200_ctx *ctx, const LpTable &t, const TablePlan &pl, CellRange cr, const double *models_dev,
                      int ld_models, int local_theta, int *nl) {
    cudaStream_t st = ctx->stream;
    const int n = cr.c1 - cr.c0;
    SCDE_CUDA(launch_row_cell(t.row_off.p, cr, t.row_cell.p, st));
    ++*nl;
    if (pl.fast) {
        SCDE_CUDA(launch_row_consts(models_dev, ld_models, t.row_off.p, cr, t.row_cell.p, t.row_x.p, pl.rowc, t.row_snap.p,
                                    pl.prep, t.K, st));
        ++*nl;
    }
    if (t.zero_base) {
        SCDE_CUDA(launch_zero_rows(t.row_off.p + cr.c0, t.row_x.p, n, t.zero_row.p + cr.c0, cr.row_cap, st));
        SCDE_CUDA(launch_lp_rows(models_dev, ld_models, cr, t.row_off.p, t.row_cell.p, t.row_x.p, pl.prep, t.K, local_theta,
                                 t.sentinel, t.table.p, t.ld, pl.rmode, 1, t.zero_row.p, nullptr, pl.rowc, t.row_snap.p, 1, pl.qf, pl.qr,
                                 st, 0, nullptr, t.zero_compact, pl.qb));
        SCDE_CUDA(launch_based_flags(t.table.p, t.ld, t.K, t.sentinel, t.zero_row.p + cr.c0, n, t.based.p + cr.c0, st,
                                     t.zero_compact ? cr.c0 : -1));
        SCDE_CUDA(launch_lp_rows(models_dev, ld_models, cr, t.row_off.p, t.row_cell.p, t.row_x.p, pl.prep, t.K, local_theta,
                                 t.sentinel, t.table.p, t.ld, pl.rmode, 2, t.zero_row.p, t.based.p, pl.rowc, t.row_snap.p,
                                 pl.q_fused ? 0 : 1, pl.qf, pl.qr, st, ctx->opt.lp_rows_kernel == 1, t.work_counter.p,
                                 t.zero_compact, pl.qb));
        *nl += 4;
    } else {
        SCDE_CUDA(launch_lp_rows(models_dev, ld_models, cr, t.row_off.p, t.row_cell.p, t.row_x.p, pl.prep, t.K, local_theta,
                                 t.sentinel, t.table.p, t.ld, pl.rmode, 0, nullptr, nullptr, pl.rowc, t.row_snap.p, 1, nullptr, nullptr,
                                 st));
        ++*nl;
    }
    return SCDE_B200_OK;
}

// rows of the table from the per-cell model rows; t.row_off / t.row_x / t.n_rows must be set
int fill_table(scde_b200_ctx *ctx, LpTable &t, const double *models_dev, int ld_models, const double *mag_dev,
               int local_theta, int sqlogit, StageTimer *tm) {
    cudaStream_t st = ctx->stream;
    TablePlan pl = plan_table(ctx, t, local_theta);
    TRY(reserve_rows(t, pl, (size_t)t.n_rows));
    int e0 = tm ? tm->begin(st) : -1;
    int nl = 1;
    TRY(prepare_cells(ctx, t, pl, models_dev, ld_models, mag_dev, local_theta, sqlogit));
    // fixed-point planes for the tcgen05 contraction: emitted by the fast row kernel itself (the FP64 rows of non-zero
    // counts are then not stored at all), by a separate pass over the FP64 table for the general kernel
    TRY(launch_table_rows(ctx, t, pl, CellRange{0, t.n_cells, (int64_t)t.n_rows}, models_dev, ld_models, local_theta, &nl));
    t.has_q = pl.q_any;
    t.f64_rows = !(pl.q_fused && t.zero_base);
    if (pl.q_any && !pl.q_fused) {
        SCDE_CUDA(launch_quantize_rows(t.table.p, t.ld, t.K, t.n_rows, t.q.p, t.qrange.p, pl.bounds ? t.qb.p : nullptr, st));
        ++nl;
    }
    if (tm) tm->end(SCDE_B200_T_LPTABLE, e0, st, nl);
    return SCDE_B200_OK;
}

// The contraction kernel of one call, resolved from the context's options once and passed down.  I8: tcgen05 on the
// fixed-point table where the data allow it, else the FP64 kernels (tiled where it applies); forced: tcgen05 or an error.
// Tiled: the FP64 DMMA kernel or an error.  Generic: the generic FP64 kernel.
enum class Contraction { I8, Tiled, Generic };
struct ContractChoice {
    Contraction kernel;
    bool forced = false;
};

ContractChoice contraction_choice(const scde_b200_ctx *ctx) {
    switch (ctx->opt.contract_kernel) {
    case 1: return {Contraction::Generic};
    case 2: return {Contraction::Tiled};
    case 3: return {Contraction::I8, true};
    default: return {Contraction::I8};
    }
}

// unique-count indices from raw counts (device, column-major, leading dimension ldc, genes [g0, g0+G)).
// known_cap > 0: the row buffers already hold known_cap rows (an earlier run of the same job) -- nothing is read back, the
// emit pass and the row kernels take their bounds from row_off on the device and stop at the capacity; the caller
// checks row_off[C] <= known_cap once the stream has drained (diff_download_impl) and repeats the run if not.
int index_from_counts(scde_b200_ctx *ctx, LpTable &t, const int32_t *counts_dev, int64_t ldc, int g0, int G, int C,
                      StageTimer *tm, int64_t known_cap = 0) {
    cudaStream_t st = ctx->stream;
    t.n_cells = C;
    t.n_genes = G;
    t.ld_ridx = C;
    SCDE_CUDA(t.n_unique.ensure(C));
    SCDE_CUDA(t.row_off.ensure((size_t)C + 1));
    SCDE_CUDA(t.err.ensure(1));
    SCDE_CUDA(t.ridx.ensure((size_t)G * C));
    int e0 = tm ? tm->begin(st) : -1;
    SCDE_CUDA(cudaMemsetAsync(t.err.p, 0, sizeof(int32_t), st));
    SCDE_CUDA(t.dedup_bits.ensure(dedup_scratch_words(C)));
    SCDE_CUDA(launch_dedup_count(counts_dev, ldc, g0, G, C, t.n_unique.p, t.err.p, t.dedup_bits.p, st));
    SCDE_CUDA(launch_exclusive_scan(t.n_unique.p, t.row_off.p, C, nullptr, st));
    int64_t cap = known_cap;
    if (known_cap <= 0) {
        int32_t total = 0, err = 0;
        SCDE_CUDA(cudaMemcpyAsync(&total, t.row_off.p + C, sizeof(int32_t), cudaMemcpyDeviceToHost, st));
        SCDE_CUDA(cudaMemcpyAsync(&err, t.err.p, sizeof(int32_t), cudaMemcpyDeviceToHost, st));
        SCDE_CUDA(cudaStreamSynchronize(st));  // the table is sized by the number of distinct (cell, count) pairs
        if (err & 1) {
            set_error("negative count in the count matrix");
            return SCDE_B200_EINVAL;
        }
        if (err & 2) {
            set_error("a cell has >= 32768 distinct count values among the processed genes (hash capacity)");
            return SCDE_B200_ELIMIT;
        }
        cap = total;
    }
    t.n_rows = cap;
    SCDE_CUDA(t.row_x.ensure((size_t)cap));
    SCDE_CUDA(launch_dedup_emit(counts_dev, ldc, g0, G, C, t.row_off.p, t.row_x.p, t.ridx.p, t.ld_ridx, t.err.p, cap,
                                t.dedup_bits.p, st));
    if (tm) tm->end(SCDE_B200_T_DEDUP, e0, st, 5);
    return SCDE_B200_OK;
}

// The device buffers of run_joint.  Joint j (W, Z, W8, zb): the j-th of the joints over the same cells that one run
// computes together.  Side i (T, SR): the i-th side of a tcgen05 launch -- side 1 is the second joint, or the second
// pass of a paired-pass launch.
struct JointScratch {
    DBuf<double> W[2], Z[2], T[2];
    DBuf<double> zpart, spart;  // base-sum and soft-max partial sums (every joint and side in turn, on one stream)
    DBuf<int8_t> W8[2];
    DBuf<uint32_t> SR[2];  // sentinel range of every (gene, boot) of one launch of the tcgen05 kernel
    DBuf<int32_t> lst_row, lst_cell, lst_len, order;
    DBuf<unsigned long long> total;  // running sums over the joints of one run: list lengths, then launch_prune_items' four
    // pruning (launch_prune_items): Z extrema of each joint, live pieces and items of one launch, and the live count
    DBuf<double> zb[2];
    DBuf<int32_t> items, n_live;
    DBuf<uint8_t> live;
};

// The big allocations of scde.expression.difference (counts shard, index matrix, lp table, joint posteriors, ratio
// posteriors).  They live in the context and are reused by successive jobs, so a one-shot call does not pay a
// cudaMalloc/cudaFree of tens of GB every time; one job per context at a time.
struct DiffWorkspace {
    DBuf<int32_t> counts;  // [C][G] (column-major shard)
    LpTable table;
    JointScratch scr;
    DBuf<double> jp[4];
    DBuf<double> post, bpost, apost;  // [G][ld] gene-major ratio posteriors
    DBuf<double> tbuf;                // transposition scratch for downloads
};

// The draw sets of a joint (DESIGN.md "Draw sets"): n sets of n_boot x D draws back to back, gene g using set
// gene_set[g] (device, NULL when n == 1).  W, W8 and Z hold one block per set ([set][pass][row]); every contraction launch
// covers all sets, each gene reading its own set's block.
struct DrawSets {
    int n = 1;
    const int32_t *gene_set = nullptr;
};

// One joint of run_joint: its draws (n_boot x D per draw set, device) and its output
struct Joint {
    const int32_t *boot_idx_dev;
    int D;
    double *jp_dev;
};

// The tcgen05 contraction of joints[0 .. n_joints) (two: joints over the same cells and entry lists with their own draws)
// whose operands run_joint has prepared.  The launches raise bits in *status (read_status).
// prune (DESIGN.md 4.3): before each launch a bound pass and a decision find the (gene, piece) items the soft-max cannot
// see; the contraction and the soft-max then skip them.  prune_stats (or NULL): launch_prune_items' four counters.
int contract_joint_i8(scde_b200_ctx *ctx, const LpTable &t, const GeneLists &lists, JointScratch &scr, int n_w_rows,
                      int n_boot, const DrawSets &sets, double scale, const Joint *joints, int n_joints, int ld_jp,
                      int hot_rank, int32_t *status, StageTimer *tm, bool prune, unsigned long long *prune_stats) {
    cudaStream_t st = ctx->stream;
    const int passes = (n_boot + WP_TILED - 1) / WP_TILED;
    ContractI8Args q{};
    q.qtable = t.q.p;
    q.ldq = q_row_bytes(t.K);
    q.row_range = t.qrange.p;
    q.lists = lists;
    q.n_w_rows = n_w_rows;
    q.n_boot = n_boot;
    q.gene_set = sets.gene_set;
    q.set_w8 = (int64_t)passes * n_w_rows * Q_WB;
    q.set_z = (int64_t)passes * WP_TILED * KP_TILED;
    q.scale = scale;
    q.sentinel = t.sentinel;
    q.K = t.K;
    q.ld_jp = ld_jp;
    q.err = status;
    q.dbg = nullptr;
    q.item_order = ctx->opt.item_order;
    q.hot_rank = hot_rank;
    q.cold_evict_first = ctx->opt.cold_evict_first;
    q.ring_stages = ctx->opt.ring_stages;
    if (ctx->opt.epilogue_timing) {
        SCDE_CUDA(ctx->epi_dbg.ensure(3));
        SCDE_CUDA(cudaMemsetAsync(ctx->epi_dbg.p, 0, 3 * sizeof(unsigned long long), st));
        q.dbg = ctx->epi_dbg.p;
    }
    // More than 104 randomizations (R's default is 150) take several passes over the same lists and rows.  Two joints
    // share every launch: (joint 0, pass ps) with (joint 1, pass ps).  One joint pairs its passes: ps with ps + 1, an odd
    // last pass on its own.
    const bool pass_pairs = n_joints == 1 && passes > 1 && ctx->opt.twin_batch_joints;
    const int n_sides = (n_joints > 1 || pass_pairs) ? 2 : 1;
    const int max_genes = contract_tiled_max_genes();
    const int mp = t.n_genes < max_genes ? t.n_genes : max_genes;
    for (int i = 0; i < n_sides; ++i) {
        SCDE_CUDA(scr.T[i].ensure(contract_tiled_scratch_doubles(t.n_genes)));
        SCDE_CUDA(scr.SR[i].ensure(contract_i8_range_words(mp)));
    }
    SCDE_CUDA(scr.spart.ensure(softmax_i8_scratch_doubles(mp)));
    if (prune) {
        for (int j = 0; j < n_joints; ++j) SCDE_CUDA(scr.zb[j].ensure(prune_zb_doubles(sets.n, n_boot)));
        SCDE_CUDA(scr.live.ensure(prune_live_bytes(mp)));
        SCDE_CUDA(scr.items.ensure((size_t)mp * q_pieces(t.K)));
        SCDE_CUDA(scr.n_live.ensure(1));
        q.qbound = t.qb.p;
        q.items = scr.items.p;  // the contraction reads the live items launch_prune_items wrote
        q.n_live = scr.n_live.p;
    }
    auto side = [&](int j, int ps, int i) {  // joint j's pass ps as side i
        return I8Side{scr.W8[j].p + (size_t)ps * n_w_rows * Q_WB, scr.Z[j].p + (size_t)ps * WP_TILED * KP_TILED, scr.T[i].p,
                      scr.SR[i].p, scr.zb[j].p, joints[j].jp_dev, ps};
    };
    struct Launch {
        I8Side s[2];
        int n;
    };
    std::vector<Launch> launches;
    for (int ps = 0; ps < passes; ++ps) {
        if (n_joints > 1)
            launches.push_back({{side(0, ps, 0), side(1, ps, 1)}, 2});
        else if (pass_pairs && ps + 1 < passes) {
            launches.push_back({{side(0, ps, 0), side(0, ps + 1, 1)}, 2});
            ++ps;
        } else
            launches.push_back({{side(0, ps, 0)}, 1});
    }
    if (prune) {
        const int e0 = tm ? tm->begin(st) : -1;
        for (int j = 0; j < n_joints; ++j) SCDE_CUDA(launch_z_bounds(q, scr.Z[j].p, sets.n, scr.zb[j].p, st));
        if (tm) tm->end(SCDE_B200_T_BOUND, e0, st, n_joints);
    }
    const uint8_t *live = prune ? scr.live.p : nullptr;
    for (int g0 = 0; g0 < t.n_genes; g0 += max_genes) {
        const int n_pos = (t.n_genes - g0) < max_genes ? (t.n_genes - g0) : max_genes;
        for (const Launch &l : launches) {
            int e0 = tm ? tm->begin(st) : -1;
            for (int i = 0; i < l.n; ++i) SCDE_CUDA(launch_sentinel_ranges(q, g0, n_pos, l.s[i], st));
            if (tm) tm->end(SCDE_B200_T_OTHER, e0, st, l.n);
            if (prune) {
                e0 = tm ? tm->begin(st) : -1;
                SCDE_CUDA(launch_prune_items(q, g0, n_pos, l.s, l.n, ctx->n_sm, scr.live.p, scr.items.p, scr.n_live.p,
                                             prune_stats, st));
                if (tm) tm->end(SCDE_B200_T_BOUND, e0, st, 2);
            }
            e0 = tm ? tm->begin(st) : -1;
            SCDE_CUDA(launch_contract_i8_pass(q, g0, n_pos, l.s, l.n, ctx->n_sm, st));
            if (tm) tm->end(SCDE_B200_T_CONTRACT, e0, st, 1);
            e0 = tm ? tm->begin(st) : -1;
            for (int i = 0; i < l.n; ++i) SCDE_CUDA(launch_softmax_i8(q, g0, n_pos, l.s[i], scr.spart.p, ctx->n_sm, st, live));
            if (tm) tm->end(SCDE_B200_T_SOFTMAX, e0, st, 2 * l.n);
        }
    }
    if (q.dbg) {
        unsigned long long h[3];
        SCDE_CUDA(cudaMemcpyAsync(h, q.dbg, sizeof(h), cudaMemcpyDeviceToHost, st));
        SCDE_CUDA(cudaStreamSynchronize(st));
        fprintf(stderr, "[scde_b200] tcgen05 epilogue: %llu items, %.0f cycles from accumulators ready to tensor memory released, "
                "MMA thread waited %.0f cycles per item for the release\n", h[1], h[1] ? (double)h[0] / h[1] : 0.0,
                h[1] ? (double)h[2] / h[1] : 0.0);
    }
    return SCDE_B200_OK;
}

// The FP64 contraction of a joint whose operands run_joint has prepared (Z = NULL outside the zero-base form)
int contract_joint_fp64(scde_b200_ctx *ctx, Contraction kernel, const LpTable &t, const GeneLists &lists,
                        JointScratch &scr, const double *Z, int n_w_rows, int n_boot, const DrawSets &sets, double scale,
                        double *jp_dev, int ld_jp, StageTimer *tm) {
    cudaStream_t st = ctx->stream;
    if (!t.f64_rows) {
        set_error("internal: the table was built in fixed point only but the FP64 contraction kernel was selected");
        return SCDE_B200_EINVAL;
    }
    ContractArgs a;
    a.table = t.table.p;
    a.ld_table = t.ld;
    a.lists = lists;
    a.W = scr.W[0].p;
    a.n_w_rows = n_w_rows;
    a.n_boot = n_boot;
    a.Z = Z;
    const int passes = (n_boot + WP_TILED - 1) / WP_TILED;
    a.gene_set = sets.gene_set;
    a.set_w_rows = (int64_t)passes * n_w_rows;
    a.set_z = (int64_t)passes * WP_TILED * t.ld;
    a.scale = scale;
    a.n_genes = t.n_genes;
    a.K = t.K;
    a.jp = jp_dev;
    a.ld_jp = ld_jp;
    a.debug = ctx->opt.debug_contract;
    const bool tiled = kernel != Contraction::Generic && contract_tiled_supported(a);
    if (kernel == Contraction::Tiled && !tiled) {
        set_error("tiled contraction kernel forced but unsupported for K=%d", t.K);
        return SCDE_B200_EINVAL;
    }
    const int e0 = tm ? tm->begin(st) : -1;
    int nl = 0;
    if (tiled) {
        SCDE_CUDA(scr.T[0].ensure(contract_tiled_scratch_doubles(t.n_genes)));
        SCDE_CUDA(launch_contract_tiled(a, ctx->n_sm, scr.T[0].p, st, &nl));
    }
    else
        SCDE_CUDA(launch_contract_generic(a, st, &nl));
    if (tm) tm->end(SCDE_B200_T_CONTRACT, e0, st, nl);
    return SCDE_B200_OK;
}

// joints[j].jp_dev[G][ld_jp] = joint posterior of the listed cells under joint j's draws, for n_joints (1 or 2) joints over
// the same cells, on the contraction kernel k selects.  Two joints share the entry lists and the launches of the tcgen05
// kernel when both can run on it and twin_batch_joints is on; otherwise they run one after the other.  The tcgen05
// launches raise bits in the device word *status, which the caller has zeroed and both joints share.
int run_joint(scde_b200_ctx *ctx, ContractChoice k, const LpTable &t, const int32_t *cell_ids_dev, int n_list,
              const Joint *joints, int n_joints, int n_boot, const DrawSets &sets, double scale, int ld_jp,
              JointScratch &scr, int32_t *status, StageTimer *tm, bool count_entries) {
    cudaStream_t st = ctx->stream;
    const int n_w_rows = round_up(n_list + 1, 16);  // at least one all-zero row after the cells (list padding)
    const int passes = (n_boot + WP_TILED - 1) / WP_TILED;
    const int ld_lst = round_up(n_list, 32);
    const bool zb = t.zero_base && t.ld <= KP_TILED;
    auto i8_for = [&](const Joint &jt) {
        return zb && t.has_q && k.kernel == Contraction::I8 && contract_i8_supported(t.K, t.ld, ld_lst, jt.D);
    };
    if (n_joints > 1 && !(i8_for(joints[0]) && i8_for(joints[1]) && ctx->opt.twin_batch_joints)) {
        for (int j = 0; j < n_joints; ++j)
            TRY(run_joint(ctx, k, t, cell_ids_dev, n_list, joints + j, 1, n_boot, sets, scale, ld_jp, scr, status, tm,
                          count_entries));
        return SCDE_B200_OK;
    }
    const bool i8 = i8_for(joints[0]);
    if (k.forced && !i8) {
        set_error("tcgen05 int8 contraction forced but unsupported here (K=%d, zero-base form %d)", t.K, (int)zb);
        return SCDE_B200_EINVAL;
    }
    const int S = sets.n;
    const size_t w_set = (size_t)passes * n_w_rows * WS_TILED, z_set = (size_t)passes * WP_TILED * t.ld;
    const size_t w8_set = (size_t)passes * n_w_rows * Q_WB;
    SCDE_CUDA(scr.lst_row.ensure((size_t)t.n_genes * ld_lst));
    SCDE_CUDA(scr.lst_cell.ensure((size_t)t.n_genes * ld_lst));
    SCDE_CUDA(scr.lst_len.ensure((size_t)t.n_genes));
    SCDE_CUDA(scr.order.ensure((size_t)t.n_genes));
    SCDE_CUDA(scr.total.ensure(5));
    if (zb) SCDE_CUDA(scr.zpart.ensure(base_sum_scratch_doubles(n_boot, t.ld)));
    for (int j = 0; j < n_joints; ++j) {
        SCDE_CUDA(scr.W[j].ensure(S * w_set));
        if (zb) SCDE_CUDA(scr.Z[j].ensure(S * z_set));
        if (i8) SCDE_CUDA(scr.W8[j].ensure(S * w8_set));
    }
    const int e0 = tm ? tm->begin(st) : -1;
    GeneLists lists{scr.lst_row.p, scr.lst_cell.p, scr.lst_len.p, scr.order.p, ld_lst};
    const int hot_rank = i8 ? ctx->opt.hot_rank : -1;  // only the tcgen05 kernel's producers know the hot bit
    SCDE_CUDA(launch_build_lists(t.ridx.p, t.ld_ridx, cell_ids_dev, n_list, t.n_genes, zb ? t.zero_row.p : nullptr,
                                 zb ? t.based.p : nullptr, 0, lists, count_entries ? scr.total.p : nullptr, st, hot_rank,
                                 n_joints));
    for (int j = 0; j < n_joints; ++j) {  // each joint's W, base sums and W8, and its output zeroed
        const Joint &jt = joints[j];
        const size_t draws_set = (size_t)n_boot * jt.D;
        for (int s = 0; s < S; ++s)
            SCDE_CUDA(launch_build_w(jt.boot_idx_dev + s * draws_set, n_boot, jt.D, n_list, scr.W[j].p + s * w_set, n_w_rows,
                                     st));
        SCDE_CUDA(cudaMemsetAsync(jt.jp_dev, 0, sizeof(double) * (size_t)t.n_genes * ld_jp, st));
        if (zb)
            for (int s = 0; s < S; ++s)
                SCDE_CUDA(launch_base_sum(t.table.p, t.ld, t.zero_row.p, t.based.p, cell_ids_dev, n_list,
                                          scr.W[j].p + s * w_set, n_w_rows, n_boot, scr.Z[j].p + s * z_set, scr.zpart.p, st,
                                          t.zero_compact));
        // W8 of all sets in one conversion: the sets' blocks are consecutive rows
        if (i8) SCDE_CUDA(launch_w_to_i8(scr.W[j].p, S * n_w_rows, n_boot, scr.W8[j].p, status, st));
    }
    // build_w is a memset and a kernel, base_sum two kernels: per extra set
    if (tm) tm->end(SCDE_B200_T_OTHER, e0, st, n_joints * ((zb ? 5 : 3) + (S - 1) * (zb ? 4 : 2)) + (i8 ? 1 : 0));
    if (!i8)
        return contract_joint_fp64(ctx, k.kernel, t, lists, scr, zb ? scr.Z[0].p : nullptr, n_w_rows, n_boot, sets, scale,
                                   joints[0].jp_dev, ld_jp, tm);
    return contract_joint_i8(ctx, t, lists, scr, n_w_rows, n_boot, sets, scale, joints, n_joints, ld_jp, hot_rank, status, tm,
                             t.has_bounds && ctx->opt.prune_pieces && n_list >= PRUNE_MIN_CELLS,
                             count_entries ? scr.total.p + 1 : nullptr);
}

// The tcgen05 status words words[0, n) once the stream has drained, copied to host[0, n).  Bits: 1 a multiplicity above
// 127; 4 a (gene, boot) whose drawn rows are "log 0" at every grid point, or a row whose "log 0" points are not the two
// ends of the grid (the FP64 kernel adds the sentinels as the reference does); 2 the pipeline watchdog.  Returns the
// watchdog's error, else SCDE_B200_OK with *rerun = whether a word asks for the FP64 kernel.
int read_status(const int32_t *words, int32_t *host, int n, bool *rerun) {
    SCDE_CUDA(cudaMemcpy(host, words, sizeof(int32_t) * n, cudaMemcpyDeviceToHost));
    int32_t any = 0;
    for (int i = 0; i < n; ++i) any |= host[i];
    if (any & 2) {
        set_error("tcgen05 contraction kernel aborted (pipeline watchdog); use scde_b200_set_contract_kernel(ctx, 2)");
        return SCDE_B200_ECUDA;
    }
    *rerun = (any & (1 | 4)) != 0;
    return SCDE_B200_OK;
}

// constant-theta fast path is valid when every cell's corr.theta is finite and positive (host check on the
// caller's model matrix, n_cells x 12 column-major with leading dimension ld)
bool theta_all_regular(const double *models, int ld, int n_cells) {
    for (int c = 0; c < n_cells; ++c) {
        const double th = models[(size_t)5 * ld + c];
        if (!(th > 0) || !std::isfinite(th)) return false;
    }
    return true;
}

std::vector<int32_t> gen_boot(int seed, int n, int n_boot) {
    std::vector<int32_t> v((size_t)n_boot * n);
    scde_b200_boot_indices(seed, n, n_boot, v.data());
    return v;
}

template <class T>
int upload(DBuf<T> &d, const T *h, size_t n, cudaStream_t st) {
    SCDE_CUDA(d.ensure(n));
    if (n) SCDE_CUDA(cudaMemcpyAsync(d.p, h, n * sizeof(T), cudaMemcpyHostToDevice, st));
    return SCDE_B200_OK;
}

int validate_index(const int32_t *v, size_t n, int lo, int hi, const char *what) {
    for (size_t i = 0; i < n; ++i)
        if (v[i] < lo || v[i] >= hi) {
            set_error("%s[%zu] = %d outside [%d, %d)", what, i, v[i], lo, hi);
            return SCDE_B200_EINVAL;
        }
    return SCDE_B200_OK;
}

// magnitudes of the prior's grid, log(max(10^x - 1, 0)) (R/functions.R:575-577)
std::vector<double> grid_magnitudes(const double *prior_x, int K) {
    std::vector<double> mag(K);
    for (int k = 0; k < K; ++k) {
        double m = std::pow(10.0, prior_x[k]) - 1;
        if (m < 0) m = 0;
        mag[k] = std::log(m);
    }
    return mag;
}

// The cells of every batch level, the pools the composition-sampled draws come from: tapply(seq_len(n) - 1, batch, I)
// (R/functions.R:570), level l's cells ascending in pool[off[l], off[l + 1]).  batch[c] < 0 = NA: the reference drops such
// a cell from every pool, as table(batch[ii]) (:356) drops it from the composition.
struct BatchPools {
    std::vector<int32_t> off, pool;
};

int batch_pools(const int32_t *batch, int C, int L, BatchPools &bp) {
    bp.off.assign(L + 1, 0);
    for (int c = 0; c < C; ++c) {
        if (batch[c] >= L) {
            set_error("batch[%d] = %d outside [0, %d) (negative = NA)", c, batch[c], L);
            return SCDE_B200_EINVAL;
        }
        if (batch[c] >= 0) bp.off[batch[c] + 1]++;
    }
    for (int l = 0; l < L; ++l) bp.off[l + 1] += bp.off[l];
    bp.pool.resize(bp.off[L] > 0 ? bp.off[L] : 1);  // (never NULL: scde_b200_batch_boot_indices checks its pointers)
    std::vector<int32_t> pos(bp.off.begin(), bp.off.end() - 1);
    for (int c = 0; c < C; ++c)
        if (batch[c] >= 0) bp.pool[pos[batch[c]]++] = c;
    return SCDE_B200_OK;
}

// table(batch[cells]) over L levels; returns D, the number of cells with a non-NA batch (draws per randomization)
int batch_composition(const int32_t *batch, int L, const int32_t *cells, size_t n, std::vector<int32_t> &comp) {
    comp.assign(L, 0);
    int D = 0;
    for (size_t i = 0; i < n; ++i)
        if (batch[cells[i]] >= 0) {
            comp[batch[cells[i]]]++;
            ++D;
        }
    return D;
}

// the entries of a zero_index with n_zero = 1 or one entry per gene that genes [g0, g0 + G) use
std::vector<int32_t> zero_slice(const int32_t *zero_index, int n_zero, int g0, int G) {
    std::vector<int32_t> zi(n_zero == 1 ? 1 : G);
    for (size_t i = 0; i < zi.size(); ++i) zi[i] = zero_index[n_zero == 1 ? 0 : g0 + i];
    return zi;
}

// One set of per-cell error models on the device (C x 12, column-major) and what building table rows from it needs
struct ModelSet {
    DBuf<double> m;
    int C = 0, local_theta = 0, sqlogit = 0;
    bool fast_theta = false;  // every corr.theta finite and > 0, no local-theta fit
};

int upload_models(ModelSet &s, const double *models, int C, int local_theta, int sqlogit, cudaStream_t st) {
    s.C = C;
    s.local_theta = local_theta;
    s.sqlogit = sqlogit;
    s.fast_theta = !local_theta && theta_all_regular(models, C, C);
    return upload(s.m, models, (size_t)C * 12, st);
}

// the table rows from the model set ms (index and row ids must be in place)
int fill_rows(scde_b200_ctx *ctx, LpTable &t, const ModelSet &ms, const double *mag_dev, StageTimer *tm) {
    t.fast_theta = ms.fast_theta;
    return fill_table(ctx, t, ms.m.p, ms.C, mag_dev, ms.local_theta, ms.sqlogit, tm);
}

// the table of a differential-expression call over C cells and a K-point grid
void init_table(const scde_b200_ctx *ctx, ContractChoice k, LpTable &t, int K, int C, bool fast_theta) {
    t.K = K;
    t.ld = table_ld(K);
    t.sentinel = -DBL_MAX / C / 1.1;
    t.fast_theta = fast_theta;
    t.zero_base = t.ld <= KP_TILED && ctx->opt.zero_base;
    t.want_q = k.kernel == Contraction::I8;
    t.want_modes = false;
}

int workspace_busy(const scde_b200_ctx *ctx) {
    if (!ctx->ws_busy) return SCDE_B200_OK;
    set_error("another expression_difference job is alive on this context (free it first)");
    return SCDE_B200_EINVAL;
}

// the context's DiffWorkspace for one job or dataset shard, held until that releases it (ctx->ws_busy = false)
int acquire_workspace(scde_b200_ctx *ctx) {
    TRY(workspace_busy(ctx));
    if (!ctx->ws) ctx->ws = new DiffWorkspace();
    ctx->ws_busy = true;
    return SCDE_B200_OK;
}

// The three ratio passes of a difference call over G genes with their shared geometry; the caller fills in the joints and
// outputs (RatioArgs' single-pair pointers, or a contrast table).
struct RatioPasses {
    RatioArgs main;      // the group joints' ratio with the prior, H0 at zero_index
    RatioArgs batch;     // batch.effect: the batch joints' ratio, default expectation = 0 (R/functions.R:362): H0 index =
                         // centre of the grid, handled in-kernel as index n (1-based) when zero_index is NULL
    RatioArgs adjusted;  // batch adjustment: the two 2K-1 posteriors slid without prior weighting (R/functions.R:391)
};

RatioPasses ratio_passes(int G, int K, int ld, const double *prior_y, const int32_t *zi, const int32_t *zi_adj, int n_zero) {
    const int nout = 2 * K - 1;
    RatioPasses r{};
    r.main.ld = ld;
    r.main.n_genes = G;
    r.main.n = K;
    r.main.prior = prior_y;
    r.main.zero_index = zi;
    r.main.n_zero = n_zero == 1 ? 1 : G;
    r.main.ld_post = round_up(nout, 8);
    r.batch = r.main;
    r.batch.zero_index = nullptr;
    r.batch.n_zero = 1;
    r.adjusted.ld = r.main.ld_post;
    r.adjusted.n_genes = G;
    r.adjusted.n = nout;
    r.adjusted.prior = nullptr;
    r.adjusted.zero_index = zi_adj;
    r.adjusted.n_zero = r.main.n_zero;
    r.adjusted.ld_post = round_up(2 * nout - 1, 8);
    return r;
}

// the main pass, and with a batch factor the batch.effect and adjusted passes after it
int launch_ratio_passes(const RatioPasses &r, bool has_batch, cudaStream_t st) {
    SCDE_CUDA(launch_ratio_summary(r.main, st));
    if (has_batch) {
        SCDE_CUDA(launch_ratio_summary(r.batch, st));
        SCDE_CUDA(launch_ratio_summary(r.adjusted, st));
    }
    return SCDE_B200_OK;
}

// Where a job's per-gene results go in the caller's (column-major) output matrices: row `row0` of matrices with `ld`
// rows.  A single-device call writes whole matrices (ld = the job's genes, row0 = 0); the shards of a multi-device call
// write their gene range of the same buffers.
struct OutPlace {
    int64_t ld, row0;
};

// a [3][G] block of grid indices and a Z vector on the device -> rows pl.row0.. of block `block` of the caller's outputs
// (blocks of pl.ld x 3 and pl.ld); a NULL destination is skipped
int download_summary(cudaStream_t st, int G, const int32_t *idx, const double *z, int32_t *idx_dst, double *z_dst,
                     OutPlace pl, size_t block = 0) {
    if (idx_dst)
        SCDE_CUDA(cudaMemcpy2DAsync(idx_dst + block * 3 * pl.ld + pl.row0, sizeof(int32_t) * (size_t)pl.ld, idx,
                                    sizeof(int32_t) * (size_t)G, sizeof(int32_t) * (size_t)G, 3, cudaMemcpyDeviceToHost, st));
    if (z_dst)
        SCDE_CUDA(cudaMemcpyAsync(z_dst + block * pl.ld + pl.row0, z, sizeof(double) * (size_t)G, cudaMemcpyDeviceToHost, st));
    return SCDE_B200_OK;
}

// stage times and launches of the timer, the table's rows and the list entries the joints contracted (the stream has
// drained)
int collect_stats(StageTimer &tm, const DiffWorkspace *ws, scde_b200_stats *stats) {
    if (!stats) return SCDE_B200_OK;
    tm.collect(stats);
    stats->table_rows = ws->table.n_rows;
    unsigned long long tot[5] = {0, 0, 0, 0, 0};
    SCDE_CUDA(cudaMemcpy(tot, ws->scr.total.p, sizeof(tot), cudaMemcpyDeviceToHost));
    stats->contract_cells = (int64_t)tot[0];
    stats->prune_items = (int64_t)tot[1];
    stats->prune_live = (int64_t)tot[2];
    stats->prune_work = (int64_t)tot[3];
    stats->prune_live_work = (int64_t)tot[4];
    return SCDE_B200_OK;
}

// Benjamini-Hochberg cZ over the n genes of result block `block` for every Z whose cZ the caller asked for
template <class Out>
void bh_outputs(const Out *o, bool has_batch, int n, size_t block = 0) {
    const size_t off = block * n;
    if (o->cz) scde::bh_cz(o->z + off, n, o->cz + off);
    if (has_batch && o->batch_cz) scde::bh_cz(o->batch_z + off, n, o->batch_cz + off);
    if (has_batch && o->adjusted_cz) scde::bh_cz(o->adjusted_z + off, n, o->adjusted_cz + off);
}

// shard i of n over genes [0, N): contiguous ranges, the first N % n of them one gene longer
void shard_range(int N, int n, int i, int *b, int *e) {
    const int base = N / n, rem = N % n;
    *b = i * base + (i < rem ? i : rem);
    *e = *b + base + (i < rem ? 1 : 0);
}

// The draw sets a call or shard over genes [g0, g1) of N holds (DESIGN.md "Draw sets"): the reference's n.cores = n splits
// [0, N) into n chunks (shard_range, R/functions.R:606-617) when n > 1 and N > n, and chunk i = [b_i, e_i) draws with
// Seed = seed + b_i; otherwise one set from `seed`.  The sets are the chunks that meet [g0, g1), in order.
struct DrawChunks {
    int first = 0;                  // global index of the first set's chunk
    std::vector<int32_t> seeds;     // one per set
    std::vector<int32_t> gene_set;  // per gene of [g0, g1): its set; empty with one set
    int n_sets() const { return (int)seeds.size(); }
};

int check_draw_chunks(int32_t n, bool explicit_draws, const char *who) {
    if (n < 0) {
        set_error("%s: draw_chunks %d < 0", who, n);
        return SCDE_B200_EINVAL;
    }
    if (n > SCDE_B200_MAX_DRAW_CHUNKS) {
        set_error("%s: draw_chunks %d above SCDE_B200_MAX_DRAW_CHUNKS (%d)", who, n, SCDE_B200_MAX_DRAW_CHUNKS);
        return SCDE_B200_ELIMIT;
    }
    if (n > 1 && explicit_draws) {
        set_error("%s: draw_chunks > 1 draws every gene chunk from its own seed; it cannot be combined with explicit boot_idx",
                  who);
        return SCDE_B200_EINVAL;
    }
    return SCDE_B200_OK;
}

// the seeds of all draw sets over genes [0, N), in chunk order
std::vector<int32_t> chunk_seeds(int N, int n, int seed) {
    if (!(n > 1 && N > n)) return {seed};
    std::vector<int32_t> v(n);
    for (int i = 0; i < n; ++i) {
        int b = 0, e = 0;
        shard_range(N, n, i, &b, &e);
        v[i] = seed + b;
    }
    return v;
}

DrawChunks draw_chunks_of(int N, int n, int seed, int g0, int g1) {
    DrawChunks d;
    if (!(n > 1 && N > n)) {
        d.seeds.push_back(seed);
        return d;
    }
    for (int i = 0; i < n; ++i) {
        int b = 0, e = 0;
        shard_range(N, n, i, &b, &e);
        if (e <= g0 || b >= g1) continue;
        if (d.seeds.empty()) d.first = i;
        const int set = d.n_sets();
        d.seeds.push_back(seed + b);
        for (int g = b > g0 ? b : g0; g < (e < g1 ? e : g1); ++g) d.gene_set.push_back(set);
    }
    if (d.n_sets() == 1) d.gene_set.clear();
    return d;
}

// Helper threads of parallel_for alive in the process.  Concurrent calls (one per device shard of a multi-device context)
// share one budget of hardware_concurrency() - 1 helpers, so they never oversubscribe the host together.
std::atomic<int> g_helper_threads{0};

// Runs f(i) for i < n on the calling thread plus as many helper threads as the process-wide budget allows (none when
// n <= 1 or the budget is spent: the calling thread then runs every task); f returns a status, the first failure (in
// task order) is returned.  A helper thread that cannot be started is simply not used.  The draw sets of a call are
// independent: they are generated in parallel.
template <class F>
int parallel_for(int n, F f) {
    if (n <= 0) return SCDE_B200_OK;
    if (n == 1) return f(0);
    std::atomic<int> next{0};
    std::vector<int> rc(n, SCDE_B200_OK);
    std::vector<std::string> msg(n);
    auto worker = [&] {
        for (int i; (i = next.fetch_add(1)) < n;)
            if ((rc[i] = f(i)) != SCDE_B200_OK) msg[i] = g_err;  // the error text is thread-local
    };
    const int hw = std::thread::hardware_concurrency() > 0 ? (int)std::thread::hardware_concurrency() : 1;
    const int want = (n < hw ? n : hw) - 1;
    int reserved = 0;
    while (reserved < want) {
        int cur = g_helper_threads.load();
        if (cur >= hw - 1) break;
        if (g_helper_threads.compare_exchange_weak(cur, cur + 1)) ++reserved;
    }
    std::vector<std::thread> th;
    try {
        th.reserve(reserved);
        for (int i = 0; i < reserved; ++i) th.emplace_back(worker);
    } catch (...) {  // no further helpers: the started ones and the calling thread share the tasks
    }
    worker();
    for (auto &t : th) t.join();
    g_helper_threads.fetch_sub(reserved);
    for (int i = 0; i < n; ++i)
        if (rc[i] != SCDE_B200_OK) {
            g_err = msg[i];
            return rc[i];
        }
    return SCDE_B200_OK;
}

// Runs f(i) for i < n on one host thread each (directly when n == 1); exceptions become return codes, the first failing
// shard's error text becomes this thread's.
template <class F>
int on_shards(int n, const std::vector<scde_b200_ctx *> &devs, F f, std::vector<scde_b200_stats> *sst, scde_b200_stats *stats) {
    std::vector<int> rc(n, SCDE_B200_OK);
    std::vector<std::string> msg(n);
    auto body = [&](int i) {
        try {
            rc[i] = f(i);
            if (rc[i] != SCDE_B200_OK) msg[i] = g_err;  // the error text is thread-local
        } catch (const std::bad_alloc &) {
            rc[i] = SCDE_B200_ENOMEM;
            msg[i] = "host allocation failed";
        } catch (const std::exception &ex) {
            rc[i] = SCDE_B200_EINVAL;
            msg[i] = ex.what();
        } catch (...) {
            rc[i] = SCDE_B200_EINVAL;
            msg[i] = "unknown exception";
        }
    };
    if (n == 1) {
        body(0);
    } else {
        std::vector<std::thread> th;
        try {
            for (int i = 0; i < n; ++i) th.emplace_back(body, i);
        } catch (...) {
            for (auto &t : th) t.join();
            set_error("could not start a host thread per device");
            return SCDE_B200_ENOMEM;
        }
        for (auto &t : th) t.join();
    }
    cudaSetDevice(devs[0]->device);
    for (int i = 0; i < n; ++i)
        if (rc[i] != SCDE_B200_OK) {
            if (n == 1)
                g_err = msg[i];
            else
                set_error("device %d (shard %d of %d): %s", devs[i]->device, i, n, msg[i].c_str());
            return rc[i];
        }
    if (stats && sst) {  // stage times: the slowest shard; counters: summed
        memset(stats, 0, sizeof(*stats));
        for (int i = 0; i < n; ++i) {
            for (int k = 0; k < SCDE_B200_T_COUNT; ++k) {
                if ((*sst)[i].ms[k] > stats->ms[k]) stats->ms[k] = (*sst)[i].ms[k];
                stats->launches[k] += (*sst)[i].launches[k];
            }
            stats->table_rows += (*sst)[i].table_rows;
            stats->contract_cells += (*sst)[i].contract_cells;
            stats->prune_items += (*sst)[i].prune_items;
            stats->prune_live += (*sst)[i].prune_live;
            stats->prune_work += (*sst)[i].prune_work;
            stats->prune_live_work += (*sst)[i].prune_live_work;
        }
    }
    return SCDE_B200_OK;
}

std::vector<scde_b200_ctx *> context_devices(scde_b200_ctx *ctx) {
    std::vector<scde_b200_ctx *> devs{ctx};
    for (auto *c : ctx->children) devs.push_back(c);
    return devs;
}

}  // namespace

// ============================================================================================
extern "C" {

int scde_b200_version(void) { return SCDE_B200_VERSION; }
const char *scde_b200_last_error(void) { return g_err.c_str(); }

int scde_b200_device_count(void) {
    int n = 0;
    if (cudaGetDeviceCount(&n) != cudaSuccess) {
        cudaGetLastError();
        return 0;
    }
    return n;
}

int scde_b200_create(int device, scde_b200_ctx **out) {
    if (!out) return SCDE_B200_EINVAL;
    *out = nullptr;
    int n = scde_b200_device_count();
    if (n <= 0) {
        set_error("no CUDA device available (libscde_b200 has no CPU fallback)");
        return SCDE_B200_ENODEVICE;
    }
    if (device < 0 || device >= n) {
        set_error("device %d out of range (have %d)", device, n);
        return SCDE_B200_EINVAL;
    }
    SCDE_CUDA(cudaSetDevice(device));
    cudaDeviceProp prop;
    SCDE_CUDA(cudaGetDeviceProperties(&prop, device));
    if (prop.major < 10) {
        set_error("device %d is sm_%d%d; libscde_b200 is built for sm_100a only", device, prop.major, prop.minor);
        return SCDE_B200_ENODEVICE;
    }
    scde_b200_ctx *c = new scde_b200_ctx();
    c->device = device;
    c->n_sm = prop.multiProcessorCount;
    cudaError_t e = cudaStreamCreateWithFlags(&c->stream, cudaStreamNonBlocking);
    if (e != cudaSuccess) {
        delete c;
        return cuda_fail(e, "cudaStreamCreateWithFlags", __FILE__, __LINE__);
    }
    *out = c;
    return SCDE_B200_OK;
}

void scde_b200_destroy(scde_b200_ctx *ctx) {
    if (!ctx) return;
    for (auto *c : ctx->children) scde_b200_destroy(c);
    ctx->children.clear();
    cudaSetDevice(ctx->device);
    if (ctx->stream) cudaStreamSynchronize(ctx->stream);
    if (ctx->copy_stream) {
        cudaStreamSynchronize(ctx->copy_stream);
        cudaStreamDestroy(ctx->copy_stream);
    }
    for (auto e : ctx->copy_events) cudaEventDestroy(e);
    if (ctx->h_draws) cudaFreeHost(ctx->h_draws);
    if (ctx->stream) cudaStreamDestroy(ctx->stream);
    delete ctx->ws;
    delete ctx;
}

void *scde_b200_stream(scde_b200_ctx *ctx) { return ctx ? (void *)ctx->stream : nullptr; }

int scde_b200_synchronize(scde_b200_ctx *ctx) {
    CHECK_CTX(ctx);
    SCDE_CUDA(cudaStreamSynchronize(ctx->stream));
    return SCDE_B200_OK;
}

int scde_b200_set_contract_kernel(scde_b200_ctx *ctx, int32_t which) {
    if (!ctx || which < 0 || which > 3) return SCDE_B200_EINVAL;
    ctx->opt.contract_kernel = which;
    for (auto *c : ctx->children) c->opt.contract_kernel = which;
    return SCDE_B200_OK;
}

int scde_b200_get_options(const scde_b200_ctx *ctx, scde_b200_options *opt) {
    if (!opt) return SCDE_B200_EINVAL;
    *opt = ctx ? ctx->opt : default_options();
    return SCDE_B200_OK;
}

int scde_b200_set_options(scde_b200_ctx *ctx, const scde_b200_options *opt) {
    if (!ctx || !opt) return SCDE_B200_EINVAL;
    if (opt->contract_kernel < 0 || opt->contract_kernel > 3 || opt->count_chunks < 0 || opt->count_chunks > 64 ||
        opt->item_order < 0 || opt->item_order > 1 ||
        !(opt->ring_stages == 0 || opt->ring_stages == 7 || opt->ring_stages == 8 || opt->ring_stages == 10)) {
        set_error("set_options: value out of range");
        return SCDE_B200_EINVAL;
    }
    ctx->opt = *opt;
    for (auto *c : ctx->children) c->opt = *opt;
    return SCDE_B200_OK;
}

int scde_b200_n_devices(const scde_b200_ctx *ctx) { return ctx ? 1 + (int)ctx->children.size() : 0; }

int scde_b200_create_multi(int n_devices, const int *devices, scde_b200_ctx **out) {
    if (!out) return SCDE_B200_EINVAL;
    *out = nullptr;
    if (n_devices < 1) {
        set_error("create_multi: n_devices must be >= 1");
        return SCDE_B200_EINVAL;
    }
    for (int i = 0; i < n_devices; ++i)
        for (int k = 0; k < i; ++k)
            if (devices && devices[i] == devices[k]) {
                set_error("create_multi: device %d listed twice", devices[i]);
                return SCDE_B200_EINVAL;
            }
    scde_b200_ctx *parent = nullptr;
    TRY(scde_b200_create(devices ? devices[0] : 0, &parent));
    for (int i = 1; i < n_devices; ++i) {
        scde_b200_ctx *c = nullptr;
        const int r = scde_b200_create(devices ? devices[i] : i, &c);
        if (r != SCDE_B200_OK) {
            scde_b200_destroy(parent);
            return r;
        }
        parent->children.push_back(c);
    }
    cudaSetDevice(parent->device);
    *out = parent;
    return SCDE_B200_OK;
}

int scde_b200_measure_fp64_peak(scde_b200_ctx *ctx, double *tflops) {
    CHECK_CTX(ctx);
    if (!tflops) return SCDE_B200_EINVAL;
    DBuf<double> sink;
    SCDE_CUDA(sink.ensure(1));
    const int iters = 20000, blocks = ctx->n_sm * 8;
    cudaEvent_t e0, e1;
    SCDE_CUDA(cudaEventCreate(&e0));
    SCDE_CUDA(cudaEventCreate(&e1));
    double best = 0;
    for (int rep = 0; rep < 4; ++rep) {
        SCDE_CUDA(cudaEventRecord(e0, ctx->stream));
        SCDE_CUDA(launch_fp64_peak(sink.p, iters, blocks, ctx->stream));
        SCDE_CUDA(cudaEventRecord(e1, ctx->stream));
        SCDE_CUDA(cudaEventSynchronize(e1));
        float ms = 0;
        SCDE_CUDA(cudaEventElapsedTime(&ms, e0, e1));
        double fl = 2.0 * 16 * (double)iters * 256 * blocks;
        double tf = fl / (ms * 1e-3) / 1e12;
        if (rep > 0 && tf > best) best = tf;
    }
    cudaEventDestroy(e0);
    cudaEventDestroy(e1);
    *tflops = best;
    return SCDE_B200_OK;
}

// --------------------------------------------------------------------------------------------
int scde_b200_cell_table(scde_b200_ctx *ctx, const double *model_row12, const int32_t *unique_counts, int32_t n_counts,
                         const double *magnitudes, int32_t n_grid, int32_t local_theta, int32_t square_logit_conc,
                         int32_t n_cells_for_clamp, double *out, int32_t *modes) {
    CHECK_CTX(ctx);
    if (!model_row12 || !unique_counts || !magnitudes || !out || n_counts < 0 || n_grid < 1 || n_cells_for_clamp < 1) {
        set_error("cell_table: bad arguments");
        return SCDE_B200_EINVAL;
    }
    cudaStream_t st = ctx->stream;
    LpTable t;
    t.n_cells = 1;
    t.K = n_grid;
    t.ld = table_ld(n_grid);
    t.n_rows = n_counts;
    t.sentinel = -DBL_MAX / n_cells_for_clamp / 1.1;
    t.fast_theta = !local_theta && theta_all_regular(model_row12, 1, 1);
    DBuf<double> d_models, d_mag;
    TRY(upload(d_models, model_row12, 12, st));
    TRY(upload(d_mag, magnitudes, (size_t)n_grid, st));
    int32_t off[2] = {0, n_counts};
    TRY(upload(t.row_off, off, 2, st));
    TRY(upload(t.row_x, unique_counts, (size_t)n_counts, st));
    TRY(fill_table(ctx, t, d_models.p, 1, d_mag.p, local_theta, square_logit_conc, nullptr));
    if (n_counts > 0) {
        SCDE_CUDA(cudaMemcpy2DAsync(out, sizeof(double) * n_grid, t.table.p, sizeof(double) * t.ld, sizeof(double) * n_grid,
                                    n_counts, cudaMemcpyDeviceToHost, st));
        if (modes)
            SCDE_CUDA(cudaMemcpyAsync(modes, t.row_mode.p, sizeof(int32_t) * n_counts, cudaMemcpyDeviceToHost, st));
    }
    SCDE_CUDA(cudaStreamSynchronize(st));
    return SCDE_B200_OK;
}

// The table the fused path builds (fill_table in the zero-base form with fixed-point planes), copied out as it lies on the
// device: the row kernels and the quantize pass the context's options select, nothing else.
int scde_b200_probe_table(scde_b200_ctx *ctx, const double *models, int32_t n_cells, const int32_t *ucl_flat,
                          const int32_t *ucl_offsets, const double *magnitudes, int32_t n_grid, int32_t local_theta,
                          int32_t square_logit_conc, int32_t n_cells_for_clamp, int8_t *q_out, uint32_t *row_range_out,
                          int32_t *zero_row_out, int32_t *based_out, double *zero_rows_out) {
    return scde_b200_probe_table_bounds(ctx, models, n_cells, ucl_flat, ucl_offsets, magnitudes, n_grid, local_theta,
                                        square_logit_conc, n_cells_for_clamp, q_out, row_range_out, zero_row_out, based_out,
                                        zero_rows_out, nullptr);
}

int scde_b200_probe_table_bounds(scde_b200_ctx *ctx, const double *models, int32_t n_cells, const int32_t *ucl_flat,
                                 const int32_t *ucl_offsets, const double *magnitudes, int32_t n_grid, int32_t local_theta,
                                 int32_t square_logit_conc, int32_t n_cells_for_clamp, int8_t *q_out, uint32_t *row_range_out,
                                 int32_t *zero_row_out, int32_t *based_out, double *zero_rows_out, int8_t *qbound_out) {
    CHECK_CTX(ctx);
    if (!models || !ucl_flat || !ucl_offsets || !magnitudes || !q_out || !row_range_out || !zero_row_out || !based_out ||
        !zero_rows_out || n_cells < 1 || n_grid < 1 || n_cells_for_clamp < 1 || ucl_offsets[0] != 0) {
        set_error("probe_table: bad arguments");
        return SCDE_B200_EINVAL;
    }
    if (n_grid > Q_MAX_K) {
        set_error("probe_table: no fixed-point table for %d grid points (at most %d)", n_grid, Q_MAX_K);
        return SCDE_B200_EINVAL;
    }
    for (int c = 0; c < n_cells; ++c) {
        if (ucl_offsets[c + 1] < ucl_offsets[c]) {
            set_error("probe_table: ucl_offsets not monotone at cell %d", c);
            return SCDE_B200_EINVAL;
        }
        for (int r = ucl_offsets[c]; r < ucl_offsets[c + 1]; ++r)
            if (ucl_flat[r] < 0 || (r > ucl_offsets[c] && ucl_flat[r] <= ucl_flat[r - 1])) {
                set_error("probe_table: the counts of cell %d are not distinct, ascending and >= 0", c);
                return SCDE_B200_EINVAL;
            }
    }
    if (ucl_offsets[n_cells] < 1) {
        set_error("probe_table: no table rows");
        return SCDE_B200_EINVAL;
    }
    cudaStream_t st = ctx->stream;
    LpTable t;
    t.n_cells = n_cells;
    t.K = n_grid;
    t.ld = table_ld(n_grid);
    t.n_rows = ucl_offsets[n_cells];
    t.sentinel = -DBL_MAX / n_cells_for_clamp / 1.1;
    t.fast_theta = !local_theta && theta_all_regular(models, n_cells, n_cells);
    t.zero_base = true;
    t.want_q = true;
    t.want_bounds = qbound_out != nullptr;
    t.want_modes = false;
    DBuf<double> d_models, d_mag;
    TRY(upload(d_models, models, (size_t)n_cells * 12, st));
    TRY(upload(d_mag, magnitudes, (size_t)n_grid, st));
    TRY(upload(t.row_off, ucl_offsets, (size_t)n_cells + 1, st));
    TRY(upload(t.row_x, ucl_flat, (size_t)t.n_rows, st));
    TRY(fill_table(ctx, t, d_models.p, n_cells, d_mag.p, local_theta, square_logit_conc, nullptr));
    if (!t.has_q) {
        set_error("probe_table: the table was built without fixed-point planes");
        return SCDE_B200_EINVAL;
    }
    SCDE_CUDA(cudaMemcpyAsync(q_out, t.q.p, (size_t)t.n_rows * q_row_bytes(n_grid), cudaMemcpyDeviceToHost, st));
    if (qbound_out && t.has_bounds) SCDE_CUDA(cudaMemcpyAsync(qbound_out, t.qb.p, (size_t)t.n_rows * Q_BW, cudaMemcpyDeviceToHost, st));
    SCDE_CUDA(cudaMemcpyAsync(row_range_out, t.qrange.p, sizeof(uint32_t) * t.n_rows, cudaMemcpyDeviceToHost, st));
    SCDE_CUDA(cudaMemcpyAsync(zero_row_out, t.zero_row.p, sizeof(int32_t) * n_cells, cudaMemcpyDeviceToHost, st));
    SCDE_CUDA(cudaMemcpyAsync(based_out, t.based.p, sizeof(int32_t) * n_cells, cudaMemcpyDeviceToHost, st));
    SCDE_CUDA(cudaStreamSynchronize(st));
    // compact form: the FP64 table holds the zero-count row of cell c in slot c; otherwise in row zero_row[c]
    for (int c = 0; c < n_cells; ++c) {
        double *dst = zero_rows_out + (size_t)c * n_grid;
        const int zr = zero_row_out[c];
        if (zr < 0) {
            for (int k = 0; k < n_grid; ++k) dst[k] = std::nan("");
            continue;
        }
        const size_t slot = t.zero_compact ? (size_t)c : (size_t)zr;
        SCDE_CUDA(cudaMemcpyAsync(dst, t.table.p + slot * t.ld, sizeof(double) * n_grid, cudaMemcpyDeviceToHost, st));
    }
    SCDE_CUDA(cudaStreamSynchronize(st));
    return SCDE_B200_OK;
}

// --------------------------------------------------------------------------------------------
static int log_boot_impl(scde_b200_ctx *ctx, const double *models, int32_t n_cells, const int32_t *ucl_flat,
                           const int32_t *ucl_offsets, const int32_t *uci, int32_t n_genes, const double *magnitudes,
                           int32_t n_grid, int32_t n_boot, const int32_t *boot_idx, int32_t D, int32_t return_individual,
                           int32_t local_theta, int32_t square_logit_conc, int32_t ensemble, int32_t modes_flag,
                           int32_t post_flag, double *jp, double *modes, double *post, ContractChoice k, bool *rerun) {
    cudaStream_t st = ctx->stream;
    (void)return_individual;
    *rerun = false;
    if (!models || !ucl_flat || !ucl_offsets || !uci || !magnitudes || !jp || n_cells < 1 || n_genes < 0 || n_grid < 1 ||
        n_boot < 0) {
        set_error("log_boot_posterior: bad arguments");
        return SCDE_B200_EINVAL;
    }
    if (ucl_offsets[0] != 0) {
        set_error("ucl_offsets[0] must be 0");
        return SCDE_B200_EINVAL;
    }
    for (int c = 0; c < n_cells; ++c) {
        if (ucl_offsets[c + 1] < ucl_offsets[c]) {
            set_error("ucl_offsets not monotone at cell %d", c);
            return SCDE_B200_EINVAL;
        }
        const int nu = ucl_offsets[c + 1] - ucl_offsets[c];
        TRY(validate_index(uci + (size_t)c * n_genes, (size_t)n_genes, 0, nu, "uci"));
    }
    if (modes_flag && !modes) {
        set_error("modes requested but the output pointer is NULL");
        return SCDE_B200_EINVAL;
    }
    if (post_flag && !post) {
        set_error("post requested but the output pointer is NULL");
        return SCDE_B200_EINVAL;
    }
    if (n_genes == 0) return SCDE_B200_OK;
    LpTable t;
    t.n_cells = n_cells;
    t.n_genes = n_genes;
    t.K = n_grid;
    t.ld = table_ld(n_grid);
    t.ld_ridx = n_cells;
    t.n_rows = ucl_offsets[n_cells];
    const double minlogprob = -DBL_MAX / n_cells / 1.1;  // src/jpmatLogBoot.cpp:127,372
    t.sentinel = -DBL_MAX / (double)(D > n_cells ? D : n_cells) / 1.1;
    t.fast_theta = !local_theta && theta_all_regular(models, n_cells, n_cells);
    t.zero_base = !post_flag && !ensemble && t.ld <= KP_TILED && ctx->opt.zero_base;
    t.want_q = k.kernel == Contraction::I8 && n_boot > 0;
    t.want_modes = modes_flag != 0;
    DBuf<double> d_models, d_mag, d_jp, d_out, d_rs;
    DBuf<int32_t> d_uci, d_boot, status;
    SCDE_CUDA(status.ensure(1));
    SCDE_CUDA(cudaMemsetAsync(status.p, 0, sizeof(int32_t), st));
    TRY(upload(d_models, models, (size_t)n_cells * 12, st));
    TRY(upload(d_mag, magnitudes, (size_t)n_grid, st));
    TRY(upload(t.row_off, ucl_offsets, (size_t)n_cells + 1, st));
    TRY(upload(t.row_x, ucl_flat, (size_t)t.n_rows, st));
    TRY(upload(d_uci, uci, (size_t)n_genes * n_cells, st));
    SCDE_CUDA(t.ridx.ensure((size_t)n_genes * n_cells));
    SCDE_CUDA(launch_uci_to_ridx(d_uci.p, n_genes, n_cells, t.row_off.p, t.ridx.p, t.ld_ridx, st));
    TRY(fill_table(ctx, t, d_models.p, n_cells, d_mag.p, local_theta, square_logit_conc, nullptr));
    const int ld_jp = t.ld;
    SCDE_CUDA(d_jp.ensure((size_t)n_genes * ld_jp));
    JointScratch scr;
    if (ensemble) {
        SCDE_CUDA(d_rs.ensure((size_t)t.n_rows));
        SCDE_CUDA(launch_ensemble(t.table.p, t.ld, t.ridx.p, t.ld_ridx, n_cells, n_genes, n_grid, d_jp.p, ld_jp, d_rs.p,
                                  t.n_rows, st));
    } else {
        std::vector<int32_t> gen;
        int nb = n_boot, dd = D;
        double scale = (double)n_boot;
        if (n_boot == 0) {  // plain product over all cells, src/jpmatLogBoot.cpp:239-249
            gen.resize(n_cells);
            for (int c = 0; c < n_cells; ++c) gen[c] = c;
            boot_idx = gen.data();
            nb = 1;
            dd = n_cells;
            scale = 1.0;
        }
        TRY(validate_index(boot_idx, (size_t)nb * dd, 0, n_cells, "boot_idx"));
        TRY(upload(d_boot, boot_idx, (size_t)nb * dd, st));
        const Joint jt{d_boot.p, dd, d_jp.p};
        TRY(run_joint(ctx, k, t, nullptr, n_cells, &jt, 1, nb, {}, scale, ld_jp, scr, status.p, nullptr, false));
    }
    SCDE_CUDA(d_out.ensure((size_t)n_genes * n_grid));
    SCDE_CUDA(launch_transpose_out(d_jp.p, ld_jp, n_genes, n_grid, d_out.p, st));
    SCDE_CUDA(cudaMemcpyAsync(jp, d_out.p, sizeof(double) * (size_t)n_genes * n_grid, cudaMemcpyDeviceToHost, st));
    if (modes_flag) {
        DBuf<double> d_modes;
        SCDE_CUDA(d_modes.ensure((size_t)n_genes * n_cells));
        SCDE_CUDA(launch_gather_modes(t.ridx.p, t.ld_ridx, n_genes, n_cells, t.row_mode.p, d_mag.p, d_modes.p, st));
        SCDE_CUDA(cudaMemcpyAsync(modes, d_modes.p, sizeof(double) * (size_t)n_genes * n_cells, cudaMemcpyDeviceToHost, st));
        SCDE_CUDA(cudaStreamSynchronize(st));
    }
    if (post_flag) {
        DBuf<double> d_post;
        const size_t np = (size_t)n_cells * n_genes * n_grid;
        SCDE_CUDA(d_post.ensure(np));
        SCDE_CUDA(launch_gather_post(t.ridx.p, t.ld_ridx, n_genes, n_cells, t.table.p, t.ld, n_grid, t.sentinel, minlogprob,
                                     d_post.p, st));
        SCDE_CUDA(cudaMemcpyAsync(post, d_post.p, sizeof(double) * np, cudaMemcpyDeviceToHost, st));
        SCDE_CUDA(cudaStreamSynchronize(st));
    }
    SCDE_CUDA(cudaStreamSynchronize(st));
    int32_t f = 0;
    return read_status(status.p, &f, 1, rerun);
}

static int log_boot_common(scde_b200_ctx *ctx, const double *models, int32_t n_cells, const int32_t *ucl_flat,
                           const int32_t *ucl_offsets, const int32_t *uci, int32_t n_genes, const double *magnitudes,
                           int32_t n_grid, int32_t n_boot, const int32_t *boot_idx, int32_t D, int32_t return_individual,
                           int32_t local_theta, int32_t square_logit_conc, int32_t ensemble, int32_t modes_flag,
                           int32_t post_flag, double *jp, double *modes, double *post) {
    bool rerun = false;
    TRY(log_boot_impl(ctx, models, n_cells, ucl_flat, ucl_offsets, uci, n_genes, magnitudes, n_grid, n_boot, boot_idx, D,
                      return_individual, local_theta, square_logit_conc, ensemble, modes_flag, post_flag, jp, modes, post,
                      contraction_choice(ctx), &rerun));
    if (!rerun) return SCDE_B200_OK;
    // a cell drawn more than 127 times in one randomization: outside the int8 operand range
    return log_boot_impl(ctx, models, n_cells, ucl_flat, ucl_offsets, uci, n_genes, magnitudes, n_grid, n_boot, boot_idx, D,
                         return_individual, local_theta, square_logit_conc, ensemble, modes_flag, post_flag, jp, modes, post,
                         {Contraction::Tiled}, &rerun);
}

int scde_b200_log_boot_posterior(scde_b200_ctx *ctx, const double *models, int32_t n_cells, const int32_t *ucl_flat,
                                 const int32_t *ucl_offsets, const int32_t *uci, int32_t n_genes,
                                 const double *magnitudes, int32_t n_grid, int32_t n_boot, int32_t seed,
                                 const int32_t *boot_idx, int32_t return_individual, int32_t local_theta,
                                 int32_t square_logit_conc, int32_t ensemble, double *jp, double *modes, double *post) {
    CHECK_CTX(ctx);
    if (n_cells < 1 || n_boot < 0) {
        set_error("log_boot_posterior: n_cells must be >= 1 and n_boot >= 0");
        return SCDE_B200_EINVAL;
    }
    std::vector<int32_t> gen;
    if (!boot_idx && n_boot > 0 && !ensemble) {
        gen = gen_boot(seed, n_cells, n_boot);
        boot_idx = gen.data();
    }
    const int mf = (return_individual == 1 || return_individual == 3);
    const int pf = (return_individual == 2 || return_individual == 3);
    return log_boot_common(ctx, models, n_cells, ucl_flat, ucl_offsets, uci, n_genes, magnitudes, n_grid, n_boot, boot_idx,
                           n_cells, return_individual, local_theta, square_logit_conc, ensemble, mf, pf, jp, modes, post);
}

int scde_b200_log_boot_batch_posterior(scde_b200_ctx *ctx, const double *models, int32_t n_cells,
                                       const int32_t *ucl_flat, const int32_t *ucl_offsets, const int32_t *uci,
                                       int32_t n_genes, const double *magnitudes, int32_t n_grid, int32_t n_levels,
                                       const int32_t *batchil_offsets, const int32_t *batchil_cells,
                                       const int32_t *composition, int32_t n_boot, int32_t seed, const int32_t *boot_idx,
                                       int32_t return_individual, int32_t local_theta, int32_t square_logit_conc,
                                       double *jp, double *modes, double *post) {
    CHECK_CTX(ctx);
    if (n_cells < 1 || n_levels < 1 || !batchil_offsets || !batchil_cells || !composition || n_boot < 1) {
        set_error("log_boot_batch_posterior: bad arguments (the reference has no n_boot == 0 branch here)");
        return SCDE_B200_EINVAL;
    }
    int D = 0;
    for (int k = 0; k < n_levels; ++k)
        if (composition[k] > 0) D += composition[k];
    if (D < 1) {
        set_error("log_boot_batch_posterior: empty composition");
        return SCDE_B200_EINVAL;
    }
    TRY(validate_index(batchil_cells, (size_t)batchil_offsets[n_levels], 0, n_cells, "batchil"));
    std::vector<int32_t> gen;
    if (!boot_idx) {
        gen.resize((size_t)n_boot * D);
        int r = scde_b200_batch_boot_indices(seed, n_levels, batchil_offsets, batchil_cells, composition, n_boot, gen.data());
        if (r != SCDE_B200_OK) {
            set_error("log_boot_batch_posterior: a sampled batch level has an empty pool");
            return r;
        }
        boot_idx = gen.data();
    }
    const int mf = (return_individual == 1);  // src/jpmatLogBoot.cpp:441,455,501
    const int pf = (return_individual == 2 || return_individual == 3);
    return log_boot_common(ctx, models, n_cells, ucl_flat, ucl_offsets, uci, n_genes, magnitudes, n_grid, n_boot, boot_idx, D,
                           return_individual, local_theta, square_logit_conc, 0, mf, pf, jp, modes, post);
}

// --------------------------------------------------------------------------------------------
static int jpmat_common(scde_b200_ctx *ctx, const double *matl, int n_mat, int n_rows, int n_cols, int n_boot,
                        const int32_t *boot_idx, int D, double *jp) {
    cudaStream_t st = ctx->stream;
    if (!matl || !jp || n_mat < 1 || n_rows < 0 || n_cols < 1 || n_boot < 0) {
        set_error("jpmat_log_boot: bad arguments");
        return SCDE_B200_EINVAL;
    }
    if (n_rows == 0) return SCDE_B200_OK;
    if ((int64_t)n_mat * n_rows > 0x7fffffffll) {  // table rows are addressed with 32-bit ids
        set_error("jpmat_log_boot: n_mat * n_rows = %lld exceeds 2^31 - 1", (long long)n_mat * n_rows);
        return SCDE_B200_ELIMIT;
    }
    TRY(validate_index(boot_idx, (size_t)n_boot * D, 0, n_mat, "boot_idx"));
    LpTable t;
    t.n_cells = n_mat;
    t.n_genes = n_rows;
    t.K = n_cols;
    t.ld = table_ld(n_cols);
    t.ld_ridx = n_mat;
    t.n_rows = (int64_t)n_mat * n_rows;
    const size_t sz = (size_t)n_rows * n_cols;
    DBuf<double> d_in, d_jp, d_out;
    DBuf<int32_t> d_boot;
    TRY(upload(d_in, matl, sz * n_mat, st));
    SCDE_CUDA(t.table.ensure((size_t)t.n_rows * t.ld));
    SCDE_CUDA(cudaMemsetAsync(t.table.p, 0, sizeof(double) * (size_t)t.n_rows * t.ld, st));
    for (int m = 0; m < n_mat; ++m)
        SCDE_CUDA(launch_transpose_in(d_in.p + sz * m, n_rows, n_cols, t.table.p + (size_t)m * n_rows * t.ld, t.ld, st));
    std::vector<int32_t> ridx((size_t)n_rows * n_mat);
    for (int g = 0; g < n_rows; ++g)
        for (int m = 0; m < n_mat; ++m) ridx[(size_t)g * n_mat + m] = m * n_rows + g;
    TRY(upload(t.ridx, ridx.data(), ridx.size(), st));
    TRY(upload(d_boot, boot_idx, (size_t)n_boot * D, st));
    SCDE_CUDA(d_jp.ensure((size_t)n_rows * t.ld));
    JointScratch scr;
    if (n_boot > 0) {
        // not divided by n_boot: src/jpmatLogBoot.cpp:36-38 (no fixed-point table: no tcgen05 launch, no status word)
        const Joint jt{d_boot.p, D, d_jp.p};
        TRY(run_joint(ctx, contraction_choice(ctx), t, nullptr, n_mat, &jt, 1, n_boot, {}, 1.0, t.ld, scr, nullptr, nullptr,
                      false));
    } else {
        SCDE_CUDA(cudaMemsetAsync(d_jp.p, 0, sizeof(double) * (size_t)n_rows * t.ld, st));
    }
    SCDE_CUDA(d_out.ensure(sz));
    SCDE_CUDA(launch_transpose_out(d_jp.p, t.ld, n_rows, n_cols, d_out.p, st));
    SCDE_CUDA(cudaMemcpyAsync(jp, d_out.p, sizeof(double) * sz, cudaMemcpyDeviceToHost, st));
    SCDE_CUDA(cudaStreamSynchronize(st));
    return SCDE_B200_OK;
}

int scde_b200_jpmat_log_boot(scde_b200_ctx *ctx, const double *matl, int32_t n_mat, int32_t n_rows, int32_t n_cols,
                             int32_t n_boot, int32_t seed, const int32_t *boot_idx, double *jp) {
    CHECK_CTX(ctx);
    if (n_mat < 1 || n_boot < 0) {
        set_error("jpmat_log_boot: bad arguments");
        return SCDE_B200_EINVAL;
    }
    std::vector<int32_t> gen;
    if (!boot_idx) {
        gen = gen_boot(seed, n_mat, n_boot);
        boot_idx = gen.data();
    }
    return jpmat_common(ctx, matl, n_mat, n_rows, n_cols, n_boot, boot_idx, n_mat, jp);
}

int scde_b200_jpmat_log_batch_boot(scde_b200_ctx *ctx, const double *matl, int32_t n_levels,
                                   const int32_t *pool_offsets, const int32_t *composition, int32_t n_rows,
                                   int32_t n_cols, int32_t n_boot, int32_t seed, const int32_t *boot_idx, double *jp) {
    CHECK_CTX(ctx);
    if (n_levels < 1 || !pool_offsets || !composition || n_boot < 0) {
        set_error("jpmat_log_batch_boot: bad arguments");
        return SCDE_B200_EINVAL;
    }
    const int n_mat = pool_offsets[n_levels];
    int D = 0;
    for (int k = 0; k < n_levels; ++k)
        if (composition[k] > 0) D += composition[k];
    std::vector<int32_t> gen, cells(n_mat);
    if (!boot_idx) {
        for (int i = 0; i < n_mat; ++i) cells[i] = i;
        gen.resize((size_t)n_boot * D);
        int r = scde_b200_batch_boot_indices(seed, n_levels, pool_offsets, cells.data(), composition, n_boot, gen.data());
        if (r != SCDE_B200_OK) {
            set_error("jpmat_log_batch_boot: a sampled pool is empty");
            return r;
        }
        boot_idx = gen.data();
    }
    return jpmat_common(ctx, matl, n_mat, n_rows, n_cols, n_boot, boot_idx, D, jp);
}

// --------------------------------------------------------------------------------------------
int scde_b200_mat_slide_mult(scde_b200_ctx *ctx, const double *m1, const double *m2, int32_t n_rows, int32_t n,
                             double *out) {
    CHECK_CTX(ctx);
    if (!m1 || !m2 || !out || n_rows < 0 || n < 1) {
        set_error("mat_slide_mult: bad arguments");
        return SCDE_B200_EINVAL;
    }
    if (n_rows == 0) return SCDE_B200_OK;
    cudaStream_t st = ctx->stream;
    const int nout = 2 * n - 1, ld = round_up(n, 8), ldo = round_up(nout, 8);
    DBuf<double> d_in, d1, d2, d_raw, d_out;
    const size_t sz = (size_t)n_rows * n;
    SCDE_CUDA(d_in.ensure(sz));
    SCDE_CUDA(d1.ensure((size_t)n_rows * ld));
    SCDE_CUDA(d2.ensure((size_t)n_rows * ld));
    SCDE_CUDA(cudaMemcpyAsync(d_in.p, m1, sizeof(double) * sz, cudaMemcpyHostToDevice, st));
    SCDE_CUDA(launch_transpose_in(d_in.p, n_rows, n, d1.p, ld, st));
    SCDE_CUDA(cudaMemcpyAsync(d_in.p, m2, sizeof(double) * sz, cudaMemcpyHostToDevice, st));
    SCDE_CUDA(launch_transpose_in(d_in.p, n_rows, n, d2.p, ld, st));
    SCDE_CUDA(d_raw.ensure((size_t)n_rows * ldo));
    RatioArgs a{};
    a.p1 = d1.p;
    a.p2 = d2.p;
    a.ld = ld;
    a.n_genes = n_rows;
    a.n = n;
    a.ld_post = ldo;
    a.raw = d_raw.p;
    SCDE_CUDA(launch_ratio_summary(a, st));
    SCDE_CUDA(d_out.ensure((size_t)n_rows * nout));
    SCDE_CUDA(launch_transpose_out(d_raw.p, ldo, n_rows, nout, d_out.p, st));
    SCDE_CUDA(cudaMemcpyAsync(out, d_out.p, sizeof(double) * (size_t)n_rows * nout, cudaMemcpyDeviceToHost, st));
    SCDE_CUDA(cudaStreamSynchronize(st));
    return SCDE_B200_OK;
}

int scde_b200_ratio_posterior_summary(scde_b200_ctx *ctx, const double *pmat1, const double *pmat2, int32_t n_genes,
                                      int32_t n, const double *prior_y, const int32_t *zero_index, int32_t n_zero,
                                      int32_t *idx, double *z, double *posterior) {
    CHECK_CTX(ctx);
    if (!pmat1 || !pmat2 || n_genes < 0 || n < 1 || !zero_index || (n_zero != 1 && n_zero != n_genes)) {
        set_error("ratio_posterior_summary: bad arguments");
        return SCDE_B200_EINVAL;
    }
    if (n_genes == 0) return SCDE_B200_OK;
    TRY(validate_index(zero_index, (size_t)n_zero, 1, 2 * n, "zero_index"));
    cudaStream_t st = ctx->stream;
    const int nout = 2 * n - 1, ld = round_up(n, 8), ldo = round_up(nout, 8);
    DBuf<double> d_in, d1, d2, d_prior, d_post, d_out, d_z;
    DBuf<int32_t> d_zi, d_idx;
    const size_t sz = (size_t)n_genes * n;
    SCDE_CUDA(d_in.ensure(sz));
    SCDE_CUDA(d1.ensure((size_t)n_genes * ld));
    SCDE_CUDA(d2.ensure((size_t)n_genes * ld));
    SCDE_CUDA(cudaMemcpyAsync(d_in.p, pmat1, sizeof(double) * sz, cudaMemcpyHostToDevice, st));
    SCDE_CUDA(launch_transpose_in(d_in.p, n_genes, n, d1.p, ld, st));
    SCDE_CUDA(cudaMemcpyAsync(d_in.p, pmat2, sizeof(double) * sz, cudaMemcpyHostToDevice, st));
    SCDE_CUDA(launch_transpose_in(d_in.p, n_genes, n, d2.p, ld, st));
    if (prior_y) TRY(upload(d_prior, prior_y, (size_t)n, st));
    TRY(upload(d_zi, zero_index, (size_t)n_zero, st));
    SCDE_CUDA(d_idx.ensure((size_t)3 * n_genes));
    SCDE_CUDA(d_z.ensure((size_t)n_genes));
    if (posterior) SCDE_CUDA(d_post.ensure((size_t)n_genes * ldo));
    RatioArgs a{};
    a.p1 = d1.p;
    a.p2 = d2.p;
    a.ld = ld;
    a.n_genes = n_genes;
    a.n = n;
    a.prior = prior_y ? d_prior.p : nullptr;
    a.zero_index = d_zi.p;
    a.n_zero = n_zero;
    a.idx = d_idx.p;
    a.z = d_z.p;
    a.post = posterior ? d_post.p : nullptr;
    a.ld_post = ldo;
    SCDE_CUDA(launch_ratio_summary(a, st));
    if (idx) SCDE_CUDA(cudaMemcpyAsync(idx, d_idx.p, sizeof(int32_t) * 3 * (size_t)n_genes, cudaMemcpyDeviceToHost, st));
    if (z) SCDE_CUDA(cudaMemcpyAsync(z, d_z.p, sizeof(double) * (size_t)n_genes, cudaMemcpyDeviceToHost, st));
    if (posterior) {
        SCDE_CUDA(d_out.ensure((size_t)n_genes * nout));
        SCDE_CUDA(launch_transpose_out(d_post.p, ldo, n_genes, nout, d_out.p, st));
        SCDE_CUDA(cudaMemcpyAsync(posterior, d_out.p, sizeof(double) * (size_t)n_genes * nout, cudaMemcpyDeviceToHost, st));
    }
    SCDE_CUDA(cudaStreamSynchronize(st));
    return SCDE_B200_OK;
}

int scde_b200_expression_magnitude(scde_b200_ctx *ctx, const int32_t *counts, int32_t n_genes, int32_t n_cells,
                                   const double *corr_b, const double *corr_a, double *out) {
    CHECK_CTX(ctx);
    if (!counts || !corr_b || !corr_a || !out || n_genes < 0 || n_cells < 0) {
        set_error("expression_magnitude: bad arguments");
        return SCDE_B200_EINVAL;
    }
    const size_t n = (size_t)n_genes * n_cells;
    if (n == 0) return SCDE_B200_OK;
    cudaStream_t st = ctx->stream;
    DBuf<int32_t> d_c;
    DBuf<double> d_b, d_a, d_o;
    TRY(upload(d_c, counts, n, st));
    TRY(upload(d_b, corr_b, (size_t)n_cells, st));
    TRY(upload(d_a, corr_a, (size_t)n_cells, st));
    SCDE_CUDA(d_o.ensure(n));
    SCDE_CUDA(launch_magnitude(d_c.p, (int64_t)n, n_genes, d_b.p, d_a.p, d_o.p, st));
    SCDE_CUDA(cudaMemcpyAsync(out, d_o.p, sizeof(double) * n, cudaMemcpyDeviceToHost, st));
    SCDE_CUDA(cudaStreamSynchronize(st));
    return SCDE_B200_OK;
}

int scde_b200_failure_probability(scde_b200_ctx *ctx, const double *models, int32_t n_cells, const int32_t *counts,
                                  const double *magnitudes, int32_t n_genes, int32_t square_logit_conc, double *out) {
    CHECK_CTX(ctx);
    if (!models || (!counts && !magnitudes) || !out || n_cells < 1 || n_genes < 0) {
        set_error("failure_probability: bad arguments (either magnitudes or counts should be provided)");
        return SCDE_B200_EINVAL;
    }
    const size_t n = (size_t)n_genes * n_cells;
    if (n == 0) return SCDE_B200_OK;
    cudaStream_t st = ctx->stream;
    DBuf<double> d_models, d_mag, d_out;
    DBuf<int32_t> d_counts;
    TRY(upload(d_models, models, (size_t)n_cells * 12, st));
    if (magnitudes)
        TRY(upload(d_mag, magnitudes, n, st));
    else
        TRY(upload(d_counts, counts, n, st));
    SCDE_CUDA(d_out.ensure(n));
    SCDE_CUDA(launch_failure_probability(magnitudes ? nullptr : d_counts.p, magnitudes ? d_mag.p : nullptr, (int64_t)n, n_genes,
                                         d_models.p, n_cells, square_logit_conc, d_out.p, st));
    SCDE_CUDA(cudaMemcpyAsync(out, d_out.p, sizeof(double) * n, cudaMemcpyDeviceToHost, st));
    SCDE_CUDA(cudaStreamSynchronize(st));
    return SCDE_B200_OK;
}

int scde_b200_expression_prior(scde_b200_ctx *ctx, const double *models, int32_t n_cells, const int32_t *counts,
                               int32_t n_genes, int32_t square_logit_conc, int32_t length_out, double pseudo_count, double bw,
                               double max_quantile, double max_value, double *x, double *y, double *lp, double *grid_weight) {
    CHECK_CTX(ctx);
    if (!models || !counts || !x || !y || n_cells < 1 || n_genes < 1 || length_out < 1 || !(bw > 0) ||
        !(max_quantile >= 0 && max_quantile <= 1)) {
        set_error("expression_prior: bad arguments");
        return SCDE_B200_EINVAL;
    }
    cudaStream_t st = ctx->stream;
    const int64_t n = (int64_t)n_genes * n_cells;
    DBuf<double> d_models, d_v, d_w, d_part;
    DBuf<int32_t> d_counts;
    DBuf<unsigned long long> d_scal, d_hist, d_bins;
    TRY(upload(d_models, models, (size_t)n_cells * 12, st));
    TRY(upload(d_counts, counts, (size_t)n, st));
    SCDE_CUDA(d_v.ensure((size_t)n));
    SCDE_CUDA(d_w.ensure((size_t)n));
    const int nb = prior_pass1_blocks(n);
    SCDE_CUDA(d_part.ensure((size_t)nb));
    SCDE_CUDA(d_scal.ensure(2));
    SCDE_CUDA(cudaMemsetAsync(d_scal.p, 0, 2 * sizeof(unsigned long long), st));
    SCDE_CUDA(launch_prior_pass1(d_counts.p, n, n_genes, d_models.p, n_cells, square_logit_conc, d_v.p, d_w.p, d_part.p, d_scal.p,
                                 d_scal.p + 1, st));
    std::vector<double> part((size_t)nb);
    unsigned long long scal[2] = {0, 0};
    SCDE_CUDA(cudaMemcpyAsync(part.data(), d_part.p, sizeof(double) * nb, cudaMemcpyDeviceToHost, st));
    SCDE_CUDA(cudaMemcpyAsync(scal, d_scal.p, sizeof(scal), cudaMemcpyDeviceToHost, st));
    SCDE_CUDA(cudaStreamSynchronize(st));
    long double wsum = 0;  // R's sum() accumulates in long double
    for (int i = 0; i < nb; ++i) wsum += part[i];
    const int64_t m = (int64_t)scal[1];
    if (std::isnan(max_value)) {  // quantile(x[x < Inf], p = max.quantile), type 7 (:233-236)
        if (m < 1) {
            set_error("expression_prior: no finite expression magnitude");
            return SCDE_B200_EINVAL;
        }
        if (max_quantile >= 1.0) {
            max_value = prior_key_to_double(scal[0]);
        } else {
            SCDE_CUDA(d_hist.ensure(256));
            auto kth = [&](int64_t rank, double *out) -> int {  // rank-th smallest (0-based) finite value: 8-pass radix select
                unsigned long long prefix = 0;
                for (int shift = 56; shift >= 0; shift -= 8) {
                    unsigned long long h[256];
                    SCDE_CUDA(cudaMemsetAsync(d_hist.p, 0, sizeof(h), st));
                    SCDE_CUDA(launch_select_hist(d_v.p, n, prefix, shift, d_hist.p, st));
                    SCDE_CUDA(cudaMemcpyAsync(h, d_hist.p, sizeof(h), cudaMemcpyDeviceToHost, st));
                    SCDE_CUDA(cudaStreamSynchronize(st));
                    int b = 0;
                    for (; b < 255 && rank >= (int64_t)h[b]; ++b) rank -= (int64_t)h[b];
                    prefix |= (unsigned long long)b << shift;
                }
                *out = prior_key_to_double(prefix);
                return SCDE_B200_OK;
            };
            const double index = 1 + (double)(m - 1) * max_quantile, fuzz = 4 * DBL_EPSILON;
            const double lo = std::floor(index + fuzz), hi = std::ceil(index - fuzz);
            double qlo = 0, qhi = 0;
            TRY(kth((int64_t)lo - 1, &qlo));
            double h = index - lo;
            if (std::fabs(h) < fuzz) h = 0;
            if (h != 0) {
                TRY(kth((int64_t)hi - 1, &qhi));
                max_value = (1 - h) * qlo + h * qhi;
            } else {
                max_value = qlo;
            }
        }
    }
    // density.default: n <- max(n, 512); if (n > 512) n <- 2^ceiling(log2(n)); lo <- from - 4 bw; up <- to + 4 bw
    const int n_user = 2 * length_out + 1;
    int nbin = n_user > 512 ? n_user : 512;
    if (nbin > 512) {
        int p2 = 1;
        while (p2 < nbin) p2 <<= 1;
        nbin = p2;
    }
    if (nbin > 16384) {
        set_error("expression_prior: length_out %d too large (working grid of %d points)", length_out, nbin);
        return SCDE_B200_ELIMIT;
    }
    const double from = -1 * max_value, to = max_value, lo = from - 4 * bw, up = to + 4 * bw;
    SCDE_CUDA(d_bins.ensure((size_t)nbin));
    SCDE_CUDA(cudaMemsetAsync(d_bins.p, 0, sizeof(unsigned long long) * nbin, st));
    SCDE_CUDA(launch_prior_bins(d_v.p, d_w.p, n, 1.0 / (double)wsum, lo, (up - lo) / (nbin - 1), nbin, d_bins.p, st));
    std::vector<unsigned long long> hb((size_t)nbin);
    SCDE_CUDA(cudaMemcpyAsync(hb.data(), d_bins.p, sizeof(unsigned long long) * nbin, cudaMemcpyDeviceToHost, st));
    SCDE_CUDA(cudaStreamSynchronize(st));
    std::vector<double> yb((size_t)nbin), dx((size_t)n_user), dy((size_t)n_user);
    for (int i = 0; i < nbin; ++i) yb[i] = (double)(long long)hb[i] / 4611686018427387904.0;
    density_from_bins(yb.data(), nbin, lo, up, bw, n_user, from, to, dx.data(), dy.data());
    const int K = length_out + 1;
    long double ys = 0;
    for (int k = 0; k < K; ++k) {  // :239-241
        x[k] = dx[length_out + k];
        double v = dy[length_out + k];
        if (std::isnan(v)) v = 0;
        y[k] = v + pseudo_count / n_genes;
        ys += y[k];
    }
    for (int k = 0; k < K; ++k) {
        y[k] /= (double)ys;  // :242
        if (lp) lp[k] = std::log(y[k]);  // :247
    }
    if (grid_weight) {  // :250 diff(10^c(x[1], x + c(diff(x)/2, 0)) - 1)
        double prev = std::pow(10.0, x[0]) - 1;
        for (int k = 0; k < K; ++k) {
            const double edge = x[k] + (k < K - 1 ? (x[k + 1] - x[k]) / 2 : 0);
            const double cur = std::pow(10.0, edge) - 1;
            grid_weight[k] = cur - prev;
            prev = cur;
        }
    }
    return SCDE_B200_OK;
}

int scde_b200_probe_contract_i8(scde_b200_ctx *ctx, const int8_t *qtable, int32_t n_rows, int32_t n_grid,
                                const uint32_t *row_range, const int8_t *w8, int32_t n_w_rows, const int32_t *lst_row,
                                const int32_t *lst_cell, const int32_t *lst_len, int32_t n_genes, int32_t ld_lst,
                                double *t_out, int32_t *flags_out) {
    return scde_b200_probe_prune_i8(ctx, qtable, n_rows, n_grid, row_range, nullptr, nullptr, w8, n_w_rows, lst_row, lst_cell,
                                    lst_len, n_genes, ld_lst, t_out, nullptr, nullptr, nullptr, nullptr, flags_out);
}

int scde_b200_probe_prune_i8(scde_b200_ctx *ctx, const int8_t *qtable, int32_t n_rows, int32_t n_grid,
                             const uint32_t *row_range, const int8_t *qbound, const double *z, const int8_t *w8,
                             int32_t n_w_rows, const int32_t *lst_row, const int32_t *lst_cell, const int32_t *lst_len,
                             int32_t n_genes, int32_t ld_lst, double *t_out, double *lb_out, double *ub_out,
                             uint8_t *live_out, double *exp_out, int32_t *flags_out) {
    CHECK_CTX(ctx);
    if (qbound && (!lb_out || !ub_out || !live_out)) {
        set_error("probe_prune_i8: bad arguments");
        return SCDE_B200_EINVAL;
    }
    if (!qtable || !w8 || !lst_row || !lst_cell || !lst_len || !t_out || n_rows < 1 || n_genes < 1 || n_w_rows < 1 ||
        !contract_i8_supported(n_grid, KP_TILED, ld_lst, 1) || n_genes > contract_tiled_max_genes()) {
        set_error("probe_contract_i8: bad arguments");
        return SCDE_B200_EINVAL;
    }
    for (int g = 0; g < n_genes; ++g) {
        if (lst_len[g] < 0 || lst_len[g] > ld_lst) {
            set_error("probe_contract_i8: lst_len[%d] out of range", g);
            return SCDE_B200_EINVAL;
        }
    }
    TRY(validate_index(lst_row, (size_t)n_genes * ld_lst, 0, n_rows, "lst_row"));
    TRY(validate_index(lst_cell, (size_t)n_genes * ld_lst, 0, n_w_rows, "lst_cell"));
    cudaStream_t st = ctx->stream;
    DBuf<int8_t> d_q, d_w;
    DBuf<int32_t> d_row, d_cell, d_len, status;
    DBuf<uint32_t> d_rr, d_sr;
    DBuf<double> d_t;
    const int ldq = q_row_bytes(n_grid);
    TRY(upload(d_q, qtable, (size_t)n_rows * ldq, st));
    if (row_range) TRY(upload(d_rr, row_range, (size_t)n_rows, st));
    TRY(upload(d_w, w8, (size_t)n_w_rows * Q_WB, st));
    TRY(upload(d_row, lst_row, (size_t)n_genes * ld_lst, st));
    TRY(upload(d_cell, lst_cell, (size_t)n_genes * ld_lst, st));
    TRY(upload(d_len, lst_len, (size_t)n_genes, st));
    const size_t nt = (size_t)n_genes * WP_TILED * KP_TILED;
    SCDE_CUDA(d_t.ensure(nt));
    SCDE_CUDA(d_sr.ensure(contract_i8_range_words(n_genes)));
    SCDE_CUDA(cudaMemsetAsync(d_t.p, 0, sizeof(double) * nt, st));
    SCDE_CUDA(status.ensure(1));
    SCDE_CUDA(cudaMemsetAsync(status.p, 0, sizeof(int32_t), st));
    ContractI8Args q{};
    q.qtable = d_q.p;
    q.ldq = ldq;
    q.row_range = row_range ? d_rr.p : nullptr;
    q.lists = GeneLists{d_row.p, d_cell.p, d_len.p, nullptr, ld_lst};
    q.n_w_rows = n_w_rows;
    q.n_boot = WP_TILED;
    q.scale = 1.0;
    q.sentinel = -1.0e300;
    q.K = n_grid;
    q.ld_jp = 0;
    q.err = status.p;
    q.item_order = ctx->opt.item_order;
    q.hot_rank = -1;
    q.cold_evict_first = 0;
    q.ring_stages = ctx->opt.ring_stages;
    I8Side side{d_w.p, nullptr, d_t.p, d_sr.p, nullptr, nullptr, 0};
    SCDE_CUDA(launch_sentinel_ranges(q, 0, n_genes, side, st));
    DBuf<int8_t> d_qb;
    DBuf<double> d_z, d_zb, d_lb, d_ub;
    DBuf<int32_t> d_items, d_nlive;
    DBuf<uint8_t> d_live;
    if (qbound) {  // the decision of the pruned contraction, with its bounds; T itself is contracted unpruned
        TRY(upload(d_qb, qbound, (size_t)n_rows * Q_BW, st));
        if (z) TRY(upload(d_z, z, (size_t)WP_TILED * KP_TILED, st));
        q.qbound = d_qb.p;
        SCDE_CUDA(d_zb.ensure(prune_zb_doubles(1, WP_TILED)));
        SCDE_CUDA(d_lb.ensure((size_t)n_genes * WP_TILED));
        SCDE_CUDA(d_ub.ensure((size_t)n_genes * WP_TILED * 4));
        SCDE_CUDA(d_live.ensure(prune_live_bytes(n_genes)));
        SCDE_CUDA(d_items.ensure((size_t)n_genes * q_pieces(n_grid)));
        SCDE_CUDA(d_nlive.ensure(1));
        side.zb = d_zb.p;
        SCDE_CUDA(launch_z_bounds(q, z ? d_z.p : nullptr, 1, d_zb.p, st));
        SCDE_CUDA(launch_prune_items(q, 0, n_genes, &side, 1, ctx->n_sm, d_live.p, d_items.p, d_nlive.p, nullptr, st, d_lb.p,
                                     d_ub.p));
    }
    SCDE_CUDA(launch_contract_i8_pass(q, 0, n_genes, &side, 1, ctx->n_sm, st));
    SCDE_CUDA(launch_finalize_t(q, n_genes, side, st));
    SCDE_CUDA(cudaMemcpyAsync(t_out, d_t.p, sizeof(double) * nt, cudaMemcpyDeviceToHost, st));
    if (qbound) {
        SCDE_CUDA(cudaMemcpyAsync(lb_out, d_lb.p, sizeof(double) * n_genes * WP_TILED, cudaMemcpyDeviceToHost, st));
        SCDE_CUDA(cudaMemcpyAsync(ub_out, d_ub.p, sizeof(double) * n_genes * WP_TILED * 4, cudaMemcpyDeviceToHost, st));
        SCDE_CUDA(cudaMemcpyAsync(live_out, d_live.p, n_genes, cudaMemcpyDeviceToHost, st));
    }
    if (exp_out) SCDE_CUDA(launch_exp_probe(exp_out, st));
    SCDE_CUDA(cudaStreamSynchronize(st));
    int32_t f = 0;
    bool rerun = false;
    const int r = read_status(status.p, &f, 1, &rerun);
    if (flags_out) *flags_out = f;
    return r;
}

}  // extern "C"

// ============================================================================================
// scde.expression.difference on the device (R/functions.R:304-408)
struct scde_b200_diff_job {
    int G = 0, C = 0, K = 0, n_boot = 0, n_levels = 0;
    int want_post = 0, has_batch = 0;
    int n_group[2] = {0, 0};
    int n_zero = 1;
    DiffWorkspace *ws = nullptr;
    scde_b200_ctx *owner = nullptr;
    ModelSet models;
    ModelSet bmodels;           // batch.models when they differ from models (else empty)
    DBuf<double> mag, prior_y;
    DBuf<int32_t> cell_ids[2];  // group cell lists
    DBuf<int32_t> boot[4];      // draws of each joint: one block of n_boot x D[i] per draw set
    int D[4] = {0, 0, 0, 0};
    DrawChunks chunks;          // the draw sets of the job's genes
    DBuf<int32_t> gene_set;     // chunks.gene_set on the device
    DBuf<int32_t> zi, zi_adj;
    DBuf<int32_t> idx, bidx, aidx;
    DBuf<double> z, bz, az;
    DBuf<int32_t> status;       // tcgen05 status words of the last run: group 0, group 1, the batch joints
    StageTimer timer;
    bool ran = false;
    int64_t known_rows = 0;          // table rows of the last completed run of this job (0: unknown): the next run needs no
                                     // size read-back -- same counts, same rows
    bool rows_unchecked = false;     // the last run used known_rows as the capacity; download verifies it
    int copy_chunks = 0;             // chunked H2D of the counts in flight on the context's copy stream:
    std::vector<int> copy_bounds;    // chunk i holds the cells [copy_bounds[i], copy_bounds[i + 1])
    int split_chunks = 0;            // > 0: the chunks [0, split_chunks) hold every cell of the first group, whose joint
                                     // runs before the rest of the front (so it hides the second half of the upload)
    int64_t front_cap = 0;           // row capacity chosen by the chunked front
    TablePlan front_plan;            // the front's table plan (buffers bound in its first phase)
    const int32_t *boot_ptr[4] = {nullptr, nullptr, nullptr, nullptr};  // draws as the device reads them
    std::vector<int32_t> ids[2];                 // cells of the two groups
    std::unique_ptr<int32_t[]> gen[4];           // generated draws (resident job), alive until their uploads have completed
    const scde_b200_diff_args *deferred_args = nullptr;  // one-shot call: the draws are still to be generated and uploaded
};

// Bootstrap draws of the group joints (local indices) and, with a batch factor, of the composition-sampled joints (global
// cell ids): the caller's, or generated from the seed (src/jpmatLogBoot.cpp:221,254-257 / :467-481).  The uploads are
// queued on the context stream; the host vectors live in the job.
// pinned: the draws go to the context's mapped pinned staging and are read in place (one-shot call with a split front:
// an H2D copy would queue behind the count matrix on the copy engine, and the first joint starts before that has landed).
int upload_draws(scde_b200_ctx *ctx, scde_b200_diff_job *j, const scde_b200_diff_args *a, bool pinned = false) {
    cudaStream_t st = ctx->stream;
    const int C = j->C;
    const int S = j->chunks.n_sets();  // draw sets per joint (a->boot_idx are NULL when S > 1)
    const int n_joints = j->has_batch ? 4 : 2;
    // draws per joint and the caller's explicit draws, validated
    BatchPools bp;
    std::vector<int32_t> comp[2];
    for (int i = 0; i < 2; ++i) j->D[i] = j->n_group[i];
    if (j->has_batch) {
        TRY(batch_pools(a->batch, C, a->n_batch_levels, bp));
        for (int i = 0; i < 2; ++i)
            j->D[2 + i] = batch_composition(a->batch, a->n_batch_levels, j->ids[i].data(), j->ids[i].size(), comp[i]);
    }
    for (int i = 0; i < n_joints; ++i)
        if (a->boot_idx[i] && j->D[i] > 0)
            TRY(validate_index(a->boot_idx[i], (size_t)a->n_boot * j->D[i], 0, i < 2 ? j->D[i] : C,
                               i < 2 ? "boot_idx" : "batch boot_idx"));
    // Destinations: the mapped pinned staging (read in place by the W build) or, for an upload, host buffers that are
    // not zero-filled first.  The generators write straight into them, one (joint, set) per task on parallel host
    // threads, so the one-shot call pays neither a zero-fill nor a copy of the draws before its first joint.
    int32_t *dst[4] = {nullptr, nullptr, nullptr, nullptr};
    int32_t *dev = nullptr;
    if (pinned) {
        size_t total = 0;
        for (int i = 0; i < n_joints; ++i) total += (size_t)S * a->n_boot * j->D[i];
        if (total > ctx->h_draws_cap) {
            if (ctx->h_draws) cudaFreeHost(ctx->h_draws);
            ctx->h_draws = nullptr;
            ctx->h_draws_cap = 0;
            SCDE_CUDA(cudaHostAlloc((void **)&ctx->h_draws, sizeof(int32_t) * total, cudaHostAllocMapped));
            ctx->h_draws_cap = total;
        }
        SCDE_CUDA(cudaHostGetDevicePointer((void **)&dev, ctx->h_draws, 0));
        size_t off = 0;
        for (int i = 0; i < n_joints; ++i) {
            dst[i] = ctx->h_draws + off;
            j->boot_ptr[i] = dev + off;
            off += (size_t)S * a->n_boot * j->D[i];
        }
    } else {
        for (int i = 0; i < n_joints; ++i)
            if (!a->boot_idx[i]) {
                j->gen[i].reset(new int32_t[(size_t)S * a->n_boot * j->D[i]]);
                dst[i] = j->gen[i].get();
            }
    }
    std::vector<std::pair<int, int>> tasks;  // (joint, set); an explicit set is one copy task (pinned) or none
    for (int i = 0; i < n_joints; ++i) {
        if (a->boot_idx[i]) {
            if (pinned) tasks.emplace_back(i, -1);
            continue;
        }
        for (int s = 0; s < S; ++s) tasks.emplace_back(i, s);
    }
    const std::vector<int32_t> &seeds = j->chunks.seeds;
    TRY(parallel_for((int)tasks.size(), [&](int t) -> int {
        const int i = tasks[t].first, s = tasks[t].second;
        const size_t per = (size_t)a->n_boot * j->D[i];
        if (s < 0) {
            memcpy(dst[i], a->boot_idx[i], sizeof(int32_t) * per);
            return SCDE_B200_OK;
        }
        int32_t *out = dst[i] + s * per;
        if (i < 2) return scde_b200_boot_indices(seeds[s], j->n_group[i], a->n_boot, out);
        return scde_b200_batch_boot_indices(seeds[s], a->n_batch_levels, bp.off.data(), bp.pool.data(), comp[i - 2].data(),
                                            a->n_boot, out);
    }));
    if (pinned) return SCDE_B200_OK;
    for (int i = 0; i < n_joints; ++i) {
        TRY(upload(j->boot[i], a->boot_idx[i] ? a->boot_idx[i] : dst[i], (size_t)S * a->n_boot * j->D[i], st));
        j->boot_ptr[i] = j->boot[i].p;
    }
    SCDE_CUDA(cudaStreamSynchronize(st));  // the caller's (or the job's) host arrays have been read
    return SCDE_B200_OK;
}

constexpr int N_COUNT_CHUNKS_DEFAULT = 8;
static int n_count_chunks(const scde_b200_ctx *ctx) {
    const int n = ctx->opt.count_chunks > 0 ? ctx->opt.count_chunks : N_COUNT_CHUNKS_DEFAULT;
    return n < 1 ? 1 : (n > 64 ? 64 : n);
}

// Queue the H2D of the shard's count matrix on the copy stream in N_COUNT_CHUNKS cell ranges, one event per range, so
// the 22 ms of PCIe time at config 4 run under the front kernels.
int start_count_copies(scde_b200_ctx *ctx, scde_b200_diff_job *j, const int32_t *counts_host, int64_t ld_host) {
    const int G = j->G, C = j->C;
    const int N_COUNT_CHUNKS = n_count_chunks(ctx);
    if (!ctx->copy_stream) SCDE_CUDA(cudaStreamCreateWithFlags(&ctx->copy_stream, cudaStreamNonBlocking));
    while ((int)ctx->copy_events.size() < N_COUNT_CHUNKS + 1) {
        cudaEvent_t e;
        SCDE_CUDA(cudaEventCreateWithFlags(&e, cudaEventDisableTiming));
        ctx->copy_events.push_back(e);
    }
    // the copy stream may overwrite the counts buffer only after earlier work on the compute stream is done with it
    SCDE_CUDA(cudaEventRecord(ctx->copy_events[N_COUNT_CHUNKS], ctx->stream));
    SCDE_CUDA(cudaStreamWaitEvent(ctx->copy_stream, ctx->copy_events[N_COUNT_CHUNKS], 0));
    // Chunk sizes: the front ends at max(last copy + the last chunk's kernels, first chunk's arrival + all kernels), so
    // the first and the last chunk are small (1/20 and 1/16 of the cells) and the ones between share the rest.
    // Split front: when every cell of the first group lies in the leading part of the matrix (the usual layout: cells
    // ordered by group), a chunk boundary is put right behind that group's last cell.  The first group's joint then
    // runs as soon as those chunks are processed -- under the upload of the rest, which is what bounds the call when
    // several ranks share the host's PCIe bandwidth (eight ranks: 35-50 ms for the 1.2 GB instead of 22).
    std::vector<int> &bounds = j->copy_bounds;
    bounds.assign(1, 0);
    j->split_chunks = 0;
    auto add_equal = [&](int lo, int hi, int n) {  // n chunks over [lo, hi), boundaries on multiples of 32, hi included
        n = n < 1 ? 1 : n;
        const int step = round_up((hi - lo + n - 1) / n, 32);
        for (int c = lo + step; c < hi; c += step) bounds.push_back(c);
        bounds.push_back(hi);
    };
    int split = 0;
    if (!j->ids[0].empty() && ctx->opt.split_front) {
        int last0 = 0;
        for (int c : j->ids[0]) last0 = c > last0 ? c : last0;
        split = round_up(last0 + 1, 32);
    }
    if (N_COUNT_CHUNKS >= 4 && C >= 64 * N_COUNT_CHUNKS && !ctx->opt.uniform_chunks) {
        const int first = round_up(C / 20, 32), last = round_up(C / 16, 32);
        if (split >= 2 * first && split <= C - 2 * last && split <= (C / 4) * 3) {
            int nA = (int)((double)N_COUNT_CHUNKS * split / C + 0.5);
            nA = nA < 2 ? 2 : (nA > N_COUNT_CHUNKS - 2 ? N_COUNT_CHUNKS - 2 : nA);
            bounds.push_back(first);
            add_equal(first, split, nA - 1);
            j->split_chunks = (int)bounds.size() - 1;
            add_equal(split, C - last - ((C - last) % 32), N_COUNT_CHUNKS - nA - 1);
            bounds.push_back(C);
        } else {
            const int mid = round_up((C - first - last + N_COUNT_CHUNKS - 3) / (N_COUNT_CHUNKS - 2), 32);
            bounds.push_back(first);
            for (int i = 0; i < N_COUNT_CHUNKS - 2 && bounds.back() + mid < C - last; ++i) bounds.push_back(bounds.back() + mid);
            if (bounds.back() < C - last) bounds.push_back(C - last - ((C - last) % 32));
            if (bounds.back() <= bounds[bounds.size() - 2]) bounds.pop_back();
            bounds.push_back(C);
        }
    } else {
        const int chunk = round_up((C + N_COUNT_CHUNKS - 1) / N_COUNT_CHUNKS, 32);
        for (int c0 = chunk; c0 < C; c0 += chunk) bounds.push_back(c0);
        bounds.push_back(C);
    }
    while ((int)ctx->copy_events.size() < (int)bounds.size() + 1) {
        cudaEvent_t e;
        SCDE_CUDA(cudaEventCreateWithFlags(&e, cudaEventDisableTiming));
        ctx->copy_events.push_back(e);
    }
    j->copy_chunks = 0;
    for (int n_ch = 0; n_ch + 1 < (int)bounds.size(); ++n_ch) {
        const int c0 = bounds[n_ch], n = bounds[n_ch + 1] - c0;
        // counted before it is queued: if a later call fails, the caller (fail() of diff_upload_impl) drains the copy stream
        // whenever copy_chunks != 0 -- the copy engine must not read the caller's buffer after the call has returned
        j->copy_chunks = n_ch + 1;
        SCDE_CUDA(cudaMemcpy2DAsync(j->ws->counts.p + (size_t)c0 * G, sizeof(int32_t) * G, counts_host + (size_t)c0 * ld_host,
                                    sizeof(int32_t) * (size_t)ld_host, sizeof(int32_t) * G, n, cudaMemcpyHostToDevice,
                                    ctx->copy_stream));
        SCDE_CUDA(cudaEventRecord(ctx->copy_events[n_ch], ctx->copy_stream));
    }
    return SCDE_B200_OK;
}

// the genes [g0, g1) a call processes: [gene_begin, gene_end), all of them when both are 0
static int gene_range(const scde_b200_diff_args *a, int *g0, int *g1) {
    *g0 = a->gene_begin;
    *g1 = a->gene_end;
    if (*g0 == 0 && *g1 == 0) *g1 = a->n_genes;
    if (*g0 < 0 || *g1 > a->n_genes || *g0 >= *g1) {
        set_error("gene range [%d, %d) invalid for %d genes", *g0, *g1, a->n_genes);
        return SCDE_B200_EINVAL;
    }
    return SCDE_B200_OK;
}

// defer_counts: the count matrix is not copied here (the one-shot call overlaps its upload with the table build)
static int diff_upload_impl(scde_b200_ctx *ctx, ContractChoice k, const scde_b200_diff_args *a, int32_t want_posteriors,
                            scde_b200_diff_job **out, bool defer_counts) {
    if (!a || !out) return SCDE_B200_EINVAL;
    *out = nullptr;
    if (!a->counts || !a->models || !a->prior_x || !a->prior_y || !a->group || a->n_genes < 1 || a->n_cells < 1 ||
        a->n_grid < 2 || a->n_boot < 1) {
        set_error("expression_difference: bad arguments");
        return SCDE_B200_EINVAL;
    }
    int g0 = 0, g1 = 0;
    TRY(gene_range(a, &g0, &g1));
    TRY(check_draw_chunks(a->draw_chunks, a->boot_idx[0] || a->boot_idx[1] || a->boot_idx[2] || a->boot_idx[3],
                          "expression_difference"));
    const int G = g1 - g0, C = a->n_cells, K = a->n_grid;
    std::vector<int32_t> ids[2];
    for (int c = 0; c < C; ++c)
        if (a->group[c] == 0 || a->group[c] == 1) ids[a->group[c]].push_back(c);
    if (ids[0].empty() || ids[1].empty()) {
        set_error("both groups need at least one cell");
        return SCDE_B200_EINVAL;
    }
    const bool has_batch = a->batch != nullptr && a->n_batch_levels > 1;
    if (a->n_zero != 1 && a->n_zero != a->n_genes) {
        set_error("n_zero must be 1 or n_genes");
        return SCDE_B200_EINVAL;
    }
    if (!a->zero_index || (has_batch && !a->zero_index_adjusted)) {
        set_error("zero_index (and zero_index_adjusted with batch) are required");
        return SCDE_B200_EINVAL;
    }
    cudaStream_t st = ctx->stream;
    TRY(acquire_workspace(ctx));
    scde_b200_diff_job *j = new scde_b200_diff_job();
    j->ws = ctx->ws;
    j->owner = ctx;
    auto fail = [&](int r) {
        if (j->copy_chunks) cudaStreamSynchronize(ctx->copy_stream);  // the copy engine reads the caller's buffer
        ctx->ws_busy = false;
        delete j;
        return r;
    };
#define JTRY(x)                                \
    do {                                       \
        int _r = (x);                          \
        if (_r != SCDE_B200_OK) return fail(_r); \
    } while (0)
#define JCUDA(x)                                                                    \
    do {                                                                            \
        cudaError_t _e = (x);                                                       \
        if (_e != cudaSuccess) return fail(cuda_fail(_e, #x, __FILE__, __LINE__));   \
    } while (0)
    j->G = G;
    j->C = C;
    j->K = K;
    j->n_boot = a->n_boot;
    j->want_post = want_posteriors;
    j->has_batch = has_batch;
    j->n_levels = has_batch ? a->n_batch_levels : 0;
    j->n_zero = a->n_zero;
    // counts shard: rows [g0, g1) of every column
    const bool trace = ctx->opt.trace != 0;
    const auto tu0 = std::chrono::steady_clock::now();
    JCUDA(j->ws->counts.ensure((size_t)G * C));
    const auto tu1 = std::chrono::steady_clock::now();
    if (!defer_counts)
        JCUDA(cudaMemcpy2DAsync(j->ws->counts.p, sizeof(int32_t) * G, a->counts + g0, sizeof(int32_t) * (size_t)a->n_genes,
                                sizeof(int32_t) * G, C, cudaMemcpyHostToDevice, st));
    if (trace && !defer_counts) {
        JCUDA(cudaStreamSynchronize(st));
        const auto tu2 = std::chrono::steady_clock::now();
        fprintf(stderr, "[scde_b200] upload: counts buffer %.2f ms, counts H2D (%.1f MB) %.2f ms\n",
                std::chrono::duration<double, std::milli>(tu1 - tu0).count(), sizeof(int32_t) * (double)G * C / 1e6,
                std::chrono::duration<double, std::milli>(tu2 - tu1).count());
    }
    JTRY(upload_models(j->models, a->models, C, a->local_theta, a->square_logit_conc, st));
    if (has_batch && a->batch_models && a->batch_models != a->models)
        JTRY(upload_models(j->bmodels, a->batch_models, C, a->batch_local_theta, a->batch_square_logit_conc, st));
    JTRY(upload(j->prior_y, a->prior_y, (size_t)K, st));
    const std::vector<double> mag = grid_magnitudes(a->prior_x, K);
    JTRY(upload(j->mag, mag.data(), (size_t)K, st));
    for (int i = 0; i < 2; ++i) {
        j->n_group[i] = (int)ids[i].size();
        JTRY(upload(j->cell_ids[i], ids[i].data(), ids[i].size(), st));
    }
    // draws: generated (host RNG, 1.3 ms per group at config 4) and uploaded now, or -- one-shot call -- while the front
    // kernels run (upload_draws is then called by diff_run_impl)
    j->ids[0] = ids[0];
    j->ids[1] = ids[1];
    j->chunks = draw_chunks_of(a->n_genes, a->draw_chunks, a->seed, g0, g1);
    if (j->chunks.n_sets() > 1) JTRY(upload(j->gene_set, j->chunks.gene_set.data(), j->chunks.gene_set.size(), st));
    if (defer_counts)
        j->deferred_args = a;
    else
        JTRY(upload_draws(ctx, j, a));
    {
        const std::vector<int32_t> zi = zero_slice(a->zero_index, a->n_zero, g0, G);
        JTRY(validate_index(zi.data(), zi.size(), 1, 2 * K, "zero_index"));
        JTRY(upload(j->zi, zi.data(), zi.size(), st));
        if (has_batch) {
            const std::vector<int32_t> za = zero_slice(a->zero_index_adjusted, a->n_zero, g0, G);
            JTRY(validate_index(za.data(), za.size(), 1, 4 * K - 2, "zero_index_adjusted"));
            JTRY(upload(j->zi_adj, za.data(), za.size(), st));
        }
        JCUDA(cudaStreamSynchronize(st));
    }
    const int ld = table_ld(K), nout = 2 * K - 1, ldo = round_up(nout, 8), nadj = 2 * nout - 1, lda = round_up(nadj, 8);
    for (int i = 0; i < (has_batch ? 4 : 2); ++i) JCUDA(j->ws->jp[i].ensure((size_t)G * ld));
    JCUDA(j->idx.ensure((size_t)3 * G));
    JCUDA(j->z.ensure((size_t)G));
    JCUDA(j->status.ensure(3));
    if (want_posteriors || has_batch) JCUDA(j->ws->post.ensure((size_t)G * ldo));
    if (has_batch) {
        JCUDA(j->ws->bpost.ensure((size_t)G * ldo));
        JCUDA(j->bidx.ensure((size_t)3 * G));
        JCUDA(j->bz.ensure((size_t)G));
        JCUDA(j->aidx.ensure((size_t)3 * G));
        JCUDA(j->az.ensure((size_t)G));
        if (want_posteriors) JCUDA(j->ws->apost.ensure((size_t)G * lda));
    }
    init_table(ctx, k, j->ws->table, K, C, j->models.fast_theta);  // the chunked front's table plan reads models' fast_theta
    JCUDA(cudaStreamSynchronize(st));
    // last: the small uploads above share the one H2D copy engine with these 1.2 GB and would queue behind them
    if (defer_counts) JTRY(start_count_copies(ctx, j, a->counts + g0, a->n_genes));
    *out = j;
    return SCDE_B200_OK;
#undef JTRY
#undef JCUDA
}

// Chunked front of the one-shot call: the count matrix goes up in N_CHUNKS cell ranges on the copy stream, and every
// range is deduplicated and its table rows are built on the compute stream as soon as it has landed, so the 1.2 GB H2D of
// config 4 (22 ms at PCIe rate) hides behind the row kernels.  Row offsets are chunk-local scans carried forward on the
// device; the row-level kernels read their bounds there (CellRange), so nothing waits for the host except one 4-byte read
// after the first chunk: its row count sizes the buffers (x 1.25).  If the estimate turns out too small the kernels stop
// at the capacity and *done stays false: the caller rebuilds index and table the classic way from the resident counts.
// phase 0: the chunks [0, split_chunks) -- all of them without a split; phase 1: the rest (split front only).  A phase
// returns with the compute stream idle and its rows checked against the capacity, so the caller may queue a joint on them.
static int front_chunked(scde_b200_ctx *ctx, scde_b200_diff_job *j, int phase, bool *done) {
    *done = false;
    LpTable &t = j->ws->table;
    const int G = j->G, C = j->C;
    cudaStream_t st = ctx->stream;
    StageTimer &tm = j->timer;
    t.n_cells = C;
    t.n_genes = G;
    t.ld_ridx = C;
    if (phase == 0) j->front_plan = plan_table(ctx, t, j->models.local_theta);
    TablePlan &pl = j->front_plan;  // prepare_cells and reserve_rows bind its buffers in phase 0
    // the copies are already in flight (start_count_copies); every path below waits for them on the compute stream
    const bool pipelined = pl.q_fused && t.zero_base && C >= 64 * j->copy_chunks && ctx->opt.pipeline_front;
    if (!pipelined) {
        j->split_chunks = 0;
        for (int i = 0; i < j->copy_chunks; ++i) SCDE_CUDA(cudaStreamWaitEvent(st, ctx->copy_events[i], 0));
        return SCDE_B200_OK;
    }
    const bool split = j->split_chunks > 0 && j->split_chunks < j->copy_chunks;
    const int ch_lo = phase == 0 ? 0 : j->split_chunks, ch_hi = (phase == 0 && split) ? j->split_chunks : j->copy_chunks;
    const bool last_phase = ch_hi == j->copy_chunks;
    auto drain = [&](int r) {  // never return while the copy engine may still read the caller's buffer
        cudaStreamSynchronize(ctx->copy_stream);
        return r;
    };
#define FTRY(x)                                   \
    do {                                          \
        int _r = (x);                             \
        if (_r != SCDE_B200_OK) return drain(_r); \
    } while (0)
#define FCUDA(x)                                                                    \
    do {                                                                            \
        cudaError_t _e = (x);                                                       \
        if (_e != cudaSuccess) return drain(cuda_fail(_e, #x, __FILE__, __LINE__));  \
    } while (0)
    const bool trace = ctx->opt.trace != 0;
    const auto tf0 = std::chrono::steady_clock::now();
    auto since = [&] { return std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now() - tf0).count(); };
    double tr_first = 0, tr_queued = 0, tr_draws = 0, tr_front = 0, tr_copy = 0;
    int e0 = 0;
    if (phase == 0) {
        FCUDA(t.n_unique.ensure(C));
        FCUDA(t.row_off.ensure((size_t)C + 1));
        FCUDA(t.err.ensure(1));
        FCUDA(t.ridx.ensure((size_t)G * C));
        FCUDA(t.dedup_bits.ensure(dedup_scratch_words(C)));
        FCUDA(cudaMemsetAsync(t.err.p, 0, sizeof(int32_t), st));
        e0 = tm.begin(st);
        FTRY(prepare_cells(ctx, t, pl, j->models.m.p, C, j->mag.p, j->models.local_theta, j->models.sqlogit));
        tm.end(SCDE_B200_T_LPTABLE, e0, st, 1);
        j->front_cap = 0;
    }
    int64_t cap = j->front_cap;
    // phase 1 follows the first group's joint (29 ms at config 4), by which time the rest of the matrix has landed: its
    // chunks are processed as one range (full grids, a sixth of the launches)
    const int ch_step = phase == 1 ? ch_hi - ch_lo : 1;
    for (int i = ch_lo; i < ch_hi; i += ch_step) {
        const int c0 = j->copy_bounds[i], n = j->copy_bounds[i + ch_step] - c0;
        const int32_t *cnt = j->ws->counts.p + (size_t)c0 * G;
        for (int e = i; e < i + ch_step; ++e) FCUDA(cudaStreamWaitEvent(st, ctx->copy_events[e], 0));
        e0 = tm.begin(st);
        uint32_t *bits = t.dedup_bits.p + dedup_scratch_words(c0) * (c0 > 0);
        FCUDA(launch_dedup_count(cnt, G, 0, G, n, t.n_unique.p + c0, t.err.p, bits, st));
        FCUDA(launch_exclusive_scan(t.n_unique.p + c0, t.row_off.p + c0, n, i ? t.row_off.p + c0 : nullptr, st));
        if (i == 0) {
            int32_t rows0 = 0;
            FCUDA(cudaMemcpyAsync(&rows0, t.row_off.p + n, sizeof(int32_t), cudaMemcpyDeviceToHost, st));
            FCUDA(cudaStreamSynchronize(st));
            tr_first = since();
            cap = (int64_t)((double)rows0 * C / n * 1.25) + 4096;
            const int64_t have = (int64_t)(t.q.cap / (size_t)q_row_bytes(t.K));  // a workspace from an earlier call
            if (have > cap) cap = have;
            if (cap > 0x7fffffff) cap = 0x7fffffff;
            FTRY(reserve_rows(t, pl, (size_t)cap));
            FCUDA(t.row_x.ensure((size_t)cap));
            j->front_cap = cap;
        }
        FCUDA(launch_dedup_emit(cnt, G, 0, G, n, t.row_off.p + c0, t.row_x.p, t.ridx.p + c0, t.ld_ridx, t.err.p, cap, bits,
                                st));
        tm.end(SCDE_B200_T_DEDUP, e0, st, 5);
        e0 = tm.begin(st);
        int nl = 0;
        FTRY(launch_table_rows(ctx, t, pl, CellRange{c0, c0 + n, cap}, j->models.m.p, C, j->models.local_theta, &nl));
        tm.end(SCDE_B200_T_LPTABLE, e0, st, nl);
    }
    tr_queued = since();
    if (trace && last_phase) {
        cudaStreamSynchronize(ctx->copy_stream);
        tr_copy = since();
    }
    if (j->deferred_args) {  // the bootstrap draws: host RNG work while the kernels queued above run
        const scde_b200_diff_args *da = j->deferred_args;
        j->deferred_args = nullptr;
        FTRY(upload_draws(ctx, j, da, split));
    }
    tr_draws = since();
    int32_t total = 0, err = 0;
    FCUDA(cudaMemcpyAsync(&total, t.row_off.p + j->copy_bounds[ch_hi], sizeof(int32_t), cudaMemcpyDeviceToHost, st));
    FCUDA(cudaMemcpyAsync(&err, t.err.p, sizeof(int32_t), cudaMemcpyDeviceToHost, st));
    FCUDA(cudaStreamSynchronize(st));
    if (last_phase) FCUDA(cudaStreamSynchronize(ctx->copy_stream));
    tr_front = since();
    if (trace)
        fprintf(stderr, "[scde_b200] front%s: first chunk counted %.2f ms, chunks queued %.2f, copies done %.2f, draws staged (incl. wait) %.2f, done %.2f\n",
                !split ? "" : (phase == 0 ? " (first group's chunks)" : " (rest)"), tr_first, tr_queued, tr_copy, tr_draws, tr_front);
#undef FTRY
#undef FCUDA
    if (err & 1) {
        cudaStreamSynchronize(ctx->copy_stream);
        set_error("negative count in the count matrix");
        return SCDE_B200_EINVAL;
    }
    if (err & 2) {
        cudaStreamSynchronize(ctx->copy_stream);
        set_error("a cell has >= 32768 distinct count values among the processed genes (hash capacity)");
        return SCDE_B200_ELIMIT;
    }
    if (total < 0 || (int64_t)total > cap) return SCDE_B200_OK;  // more rows than estimated: classic rebuild
    t.n_rows = total;
    t.has_q = true;
    t.f64_rows = false;
    *done = true;
    return SCDE_B200_OK;
}

static int diff_run_impl(scde_b200_ctx *ctx, scde_b200_diff_job *j, bool chunked_counts, ContractChoice k);

extern "C" {

int scde_b200_diff_upload(scde_b200_ctx *ctx, const scde_b200_diff_args *a, int32_t want_posteriors,
                          scde_b200_diff_job **out) {
    CHECK_CTX(ctx);
    return diff_upload_impl(ctx, contraction_choice(ctx), a, want_posteriors, out, false);
}

int scde_b200_diff_run(scde_b200_ctx *ctx, scde_b200_diff_job *j) {
    CHECK_CTX(ctx);
    return diff_run_impl(ctx, j, false, contraction_choice(ctx));
}

}  // extern "C"

// chunked_counts: the count matrix is arriving in cell chunks on the copy stream (one-shot call)
static int diff_run_impl(scde_b200_ctx *ctx, scde_b200_diff_job *j, bool chunked_counts, ContractChoice k) {
    if (!j) return SCDE_B200_EINVAL;
    cudaStream_t st = ctx->stream;
    StageTimer &tm = j->timer;
    tm.reset();
    SCDE_CUDA(j->ws->scr.total.ensure(5));
    SCDE_CUDA(cudaMemsetAsync(j->ws->scr.total.p, 0, 5 * sizeof(unsigned long long), st));
    const int G = j->G, C = j->C, K = j->K;
    const int ld = j->ws->table.ld;
    j->ws->table.want_q = k.kernel == Contraction::I8;
    SCDE_CUDA(cudaMemsetAsync(j->status.p, 0, 3 * sizeof(int32_t), st));
    int t_all = tm.begin(st);
    bool front_done = false, joint0_done = false;
    const DrawSets sets{j->chunks.n_sets(), j->gene_set.p};
    auto group_joint = [&](int i) {  // cells of one factor level, draws are local indices (R/functions.R:372-374)
        const Joint jt{j->boot_ptr[i], j->D[i], j->ws->jp[i].p};
        return run_joint(ctx, k, j->ws->table, j->cell_ids[i].p, j->n_group[i], &jt, 1, j->n_boot, sets, (double)j->n_boot,
                         ld, j->ws->scr, j->status.p + i, &tm, true);
    };
    if (chunked_counts) {
        TRY(front_chunked(ctx, j, 0, &front_done));
        if (front_done && j->split_chunks > 0 && j->split_chunks < j->copy_chunks) {
            // split front: every row of the first group's cells is built and within the capacity -- its joint runs
            // while the rest of the count matrix is still arriving
            TRY(group_joint(0));
            joint0_done = true;
            TRY(front_chunked(ctx, j, 1, &front_done));
            if (!front_done) {  // the table is rebuilt below: row ids change, the first joint is repeated
                joint0_done = false;
                SCDE_CUDA(cudaMemsetAsync(j->ws->scr.total.p, 0, 5 * sizeof(unsigned long long), st));
            }
        }
        if (!front_done && ctx->copy_stream) SCDE_CUDA(cudaStreamSynchronize(ctx->copy_stream));  // the counts must be resident
    }
    if (j->deferred_args) {  // not done by the chunked front (small problem or fallback)
        const scde_b200_diff_args *da = j->deferred_args;
        j->deferred_args = nullptr;
        TRY(upload_draws(ctx, j, da));
    }
    j->rows_unchecked = false;
    if (!front_done) {
        // a repeated run of a resident job: the buffers of the last run are exactly large enough, no host round trip
        const int64_t known = (!chunked_counts && k.kernel == Contraction::I8) ? j->known_rows : 0;
        TRY(index_from_counts(ctx, j->ws->table, j->ws->counts.p, G, 0, G, C, &tm, known));
        j->rows_unchecked = known > 0;
        TRY(fill_rows(ctx, j->ws->table, j->models, j->mag.p, &tm));
    }
    for (int i = 0; i < 2; ++i)
        if (!(i == 0 && joint0_done)) TRY(group_joint(i));
    // batch joints: all cells, composition-sampled draws are global cell ids (R/functions.R:355-357)
    if (j->has_batch) {
        // batch.models differ from models: the table rows are rebuilt from them (same row ids -- the counts have not
        // changed -- so the index matrix stays); the group joints above are done with the first table
        if (j->bmodels.m.p) TRY(fill_rows(ctx, j->ws->table, j->bmodels, j->mag.p, &tm));
        // the two composition-sampled joints walk the same cells and rows with different draws: one launch of the contraction
        // kernel for both, items paired on neighbouring SMs, so the table is pulled from DRAM once for the two
        const Joint batch[2] = {{j->boot_ptr[2], j->D[2], j->ws->jp[2].p}, {j->boot_ptr[3], j->D[3], j->ws->jp[3].p}};
        TRY(run_joint(ctx, k, j->ws->table, nullptr, C, batch, 2, j->n_boot, sets, (double)j->n_boot, ld, j->ws->scr,
                      j->status.p + 2, &tm, true));
    }
    const int e0 = tm.begin(st);
    RatioPasses r = ratio_passes(G, K, ld, j->prior_y.p, j->zi.p, j->zi_adj.p, j->n_zero);
    r.main.p1 = j->ws->jp[0].p;
    r.main.p2 = j->ws->jp[1].p;
    r.main.idx = j->idx.p;
    r.main.z = j->z.p;
    r.main.post = (j->want_post || j->has_batch) ? j->ws->post.p : nullptr;
    r.batch.p1 = j->ws->jp[2].p;
    r.batch.p2 = j->ws->jp[3].p;
    r.batch.idx = j->bidx.p;
    r.batch.z = j->bz.p;
    r.batch.post = j->ws->bpost.p;
    r.adjusted.p1 = j->ws->post.p;
    r.adjusted.p2 = j->ws->bpost.p;
    r.adjusted.idx = j->aidx.p;
    r.adjusted.z = j->az.p;
    r.adjusted.post = j->want_post ? j->ws->apost.p : nullptr;
    TRY(launch_ratio_passes(r, j->has_batch, st));
    tm.end(SCDE_B200_T_RATIO, e0, st, j->has_batch ? 3 : 1);
    tm.end(SCDE_B200_T_TOTAL, t_all, st, 0);
    j->ran = true;
    return SCDE_B200_OK;
}

// [G][ld_src] gene-major device matrix -> rows row0.. of a column-major host matrix with pl.ld rows
static int download_matrix(scde_b200_ctx *ctx, DiffWorkspace *ws, int G, const double *src, int ld_src, int cols, double *dst,
                           OutPlace pl) {
    cudaStream_t st = ctx->stream;
    SCDE_CUDA(ws->tbuf.ensure((size_t)G * cols));
    SCDE_CUDA(launch_transpose_out(src, ld_src, G, cols, ws->tbuf.p, st));
    SCDE_CUDA(cudaMemcpy2DAsync(dst + pl.row0, sizeof(double) * (size_t)pl.ld, ws->tbuf.p, sizeof(double) * (size_t)G,
                                sizeof(double) * (size_t)G, cols, cudaMemcpyDeviceToHost, st));
    SCDE_CUDA(cudaStreamSynchronize(st));
    return SCDE_B200_OK;
}

static int diff_download_impl(scde_b200_ctx *ctx, scde_b200_diff_job *j, const scde_b200_diff_out *o,
                              scde_b200_stats *stats, OutPlace pl, ContractChoice k) {
    if (!j || !j->ran) {
        set_error("diff_download: job has not been run");
        return SCDE_B200_EINVAL;
    }
    cudaStream_t st = ctx->stream;
    const int G = j->G, K = j->K;
    const int ld = j->ws->table.ld, nout = 2 * K - 1, ldo = round_up(nout, 8), nadj = 2 * nout - 1, lda = round_up(nadj, 8);
    {
        SCDE_CUDA(cudaStreamSynchronize(st));
        if (j->rows_unchecked) {  // the run took its row capacity from the previous run: confirm, else repeat with a read-back
            int32_t total = 0, err = 0;
            SCDE_CUDA(cudaMemcpy(&total, j->ws->table.row_off.p + j->C, sizeof(int32_t), cudaMemcpyDeviceToHost));
            SCDE_CUDA(cudaMemcpy(&err, j->ws->table.err.p, sizeof(int32_t), cudaMemcpyDeviceToHost));
            j->rows_unchecked = false;
            if (err || total < 0 || (int64_t)total > j->known_rows) {
                j->known_rows = 0;
                TRY(diff_run_impl(ctx, j, false, k));
                SCDE_CUDA(cudaStreamSynchronize(st));
            } else {
                j->ws->table.n_rows = total;
            }
        }
        j->known_rows = j->ws->table.n_rows;
        int32_t f[3];
        bool rerun = false;
        TRY(read_status(j->status.p, f, 3, &rerun));
        if (rerun) {  // a multiplicity above 127: repeat the run on the FP64 contraction kernel
            TRY(diff_run_impl(ctx, j, false, {Contraction::Tiled}));
            SCDE_CUDA(cudaStreamSynchronize(st));
        }
    }
    if (o) {
        TRY(download_summary(st, G, j->idx.p, j->z.p, o->idx, o->z, pl));
        if (j->has_batch) {
            TRY(download_summary(st, G, j->bidx.p, j->bz.p, o->batch_idx, o->batch_z, pl));
            TRY(download_summary(st, G, j->aidx.p, j->az.p, o->adjusted_idx, o->adjusted_z, pl));
        }
        SCDE_CUDA(cudaStreamSynchronize(st));
        for (int i = 0; i < 2; ++i) {
            if (o->joint_posteriors[i]) TRY(download_matrix(ctx, j->ws, j->G, j->ws->jp[i].p, ld, K, o->joint_posteriors[i], pl));
            if (j->has_batch && o->batch_joint_posteriors[i])
                TRY(download_matrix(ctx, j->ws, j->G, j->ws->jp[2 + i].p, ld, K, o->batch_joint_posteriors[i], pl));
        }
        if (o->difference_posterior) {
            if (!j->ws->post.p) {
                set_error("difference_posterior requested but the job was uploaded without want_posteriors");
                return SCDE_B200_EINVAL;
            }
            TRY(download_matrix(ctx, j->ws, j->G, j->ws->post.p, ldo, nout, o->difference_posterior, pl));
        }
        if (j->has_batch && o->batch_difference_posterior)
            TRY(download_matrix(ctx, j->ws, j->G, j->ws->bpost.p, ldo, nout, o->batch_difference_posterior, pl));
        if (j->has_batch && o->adjusted_difference_posterior) {
            if (!j->ws->apost.p) {
                set_error("adjusted posterior requested but the job was uploaded without want_posteriors");
                return SCDE_B200_EINVAL;
            }
            TRY(download_matrix(ctx, j->ws, j->G, j->ws->apost.p, lda, nadj, o->adjusted_difference_posterior, pl));
        }
    }
    SCDE_CUDA(cudaStreamSynchronize(st));
    return collect_stats(j->timer, j->ws, stats);
}

extern "C" {

int scde_b200_diff_download(scde_b200_ctx *ctx, scde_b200_diff_job *j, const scde_b200_diff_out *o, scde_b200_stats *stats) {
    CHECK_CTX(ctx);
    return diff_download_impl(ctx, j, o, stats, OutPlace{j ? j->G : 0, 0}, contraction_choice(ctx));
}

void scde_b200_diff_free(scde_b200_ctx *ctx, scde_b200_diff_job *job) {
    if (ctx) cudaSetDevice(ctx->device);
    if (job && job->owner) job->owner->ws_busy = false;
    delete job;
}

}  // extern "C"

// one device: upload (chunked, overlapped), run, download into the caller's buffers at `pl`
static int expression_difference_single(scde_b200_ctx *ctx, const scde_b200_diff_args *args, const scde_b200_diff_out *out,
                                        scde_b200_stats *stats, OutPlace pl) {
    CHECK_CTX(ctx);
    const ContractChoice k = contraction_choice(ctx);
    const int want_post = out->difference_posterior || out->adjusted_difference_posterior;
    const bool trace = ctx->opt.trace != 0;  // host wall-clock of the three phases on stderr
    auto now = [] { return std::chrono::steady_clock::now(); };
    auto ms = [](std::chrono::steady_clock::time_point a, std::chrono::steady_clock::time_point b) {
        return std::chrono::duration<double, std::milli>(b - a).count();
    };
    const auto t0 = now();
    scde_b200_diff_job *job = nullptr;
    int r = diff_upload_impl(ctx, k, args, want_post, &job, true);
    if (r != SCDE_B200_OK) return r;
    const auto t1 = now();
    r = diff_run_impl(ctx, job, true, k);
    if (r != SCDE_B200_OK && ctx->copy_stream) cudaStreamSynchronize(ctx->copy_stream);
    const auto t2 = now();
    if (r == SCDE_B200_OK) r = diff_download_impl(ctx, job, out, stats, pl, k);
    const auto t3 = now();
    scde_b200_diff_free(ctx, job);
    if (trace)
        fprintf(stderr, "[scde_b200] expression_difference (device %d): upload %.2f ms, run (queued) %.2f ms, download (incl. wait) %.2f ms, free %.2f ms\n",
                ctx->device, ms(t0, t1), ms(t1, t2), ms(t2, t3), ms(t3, now()));
    return r;
}

extern "C" {

int scde_b200_expression_difference(scde_b200_ctx *ctx, const scde_b200_diff_args *args, const scde_b200_diff_out *out,
                                    scde_b200_stats *stats) {
    CHECK_CTX(ctx);
    if (!args || !out) return SCDE_B200_EINVAL;
    if ((out->cz && !out->z) || (out->batch_cz && !out->batch_z) || (out->adjusted_cz && !out->adjusted_z)) {
        set_error("expression_difference: a cZ output needs the matching Z output");
        return SCDE_B200_EINVAL;
    }
    int g0 = 0, g1 = 0;
    TRY(gene_range(args, &g0, &g1));
    // Several devices: contiguous gene ranges, one per device.  Every shard holds the draw sets of the draw chunks it
    // meets, with their global seeds (draw_chunks_of over the call's n_genes), so the result does not depend on the number
    // of devices.  No inter-GPU traffic: every shard's results go to its rows of the caller's buffers by device-to-host
    // copies.
    const std::vector<scde_b200_ctx *> devs = context_devices(ctx);
    const int n = g1 - g0;
    const int n_use = (int)devs.size() < n ? (int)devs.size() : n;
    std::vector<scde_b200_stats> sst(n_use);
    TRY(on_shards(n_use, devs, [&](int i) -> int {
        int b = 0, e = 0;
        shard_range(n, n_use, i, &b, &e);
        scde_b200_diff_args a = *args;
        a.gene_begin = g0 + b;
        a.gene_end = g0 + e;
        return expression_difference_single(devs[i], &a, out, stats ? &sst[i] : nullptr, OutPlace{n, b});
    }, &sst, stats));
    // Benjamini-Hochberg over the genes of this call, once, on the host (all shards have landed)
    bh_outputs(out, args->batch != nullptr && args->n_batch_levels > 1, n);
    return SCDE_B200_OK;
}

}  // extern "C"

// ============================================================================================
// Many contrasts on one resident dataset.  The index and the table cover every cell, so they do not depend on the grouping;
// a group's joint depends only on its cells, the seed, n_boot and (through the draws) its size, because every
// scde.posteriors call of the reference re-seeds srand(Seed); a batch joint depends only on the composition of its group.
// A call therefore computes each named group's joint once into a bank slot, each distinct composition's batch joint once,
// and runs the ratio and summary passes of all contrasts in batched launches on the bank.

namespace {

// The host part of one contrasts call, shared by the per-device shards: which joints exist and which draws they use.
struct ContrastPlan {
    int C = 0, K = 0, N = 0;          // cells, grid points, genes of the dataset
    int n_contrasts = 0, n_boot = 0;
    bool has_batch = false, want_post = false;
    std::vector<int> slot_group;      // bank slot -> group id (only groups some contrast names)
    std::vector<int32_t> cells;       // the slots' cells back to back
    std::vector<int64_t> cell_off;    // slot -> offset into cells (n_slots + 1)
    int seed = 1, draw_chunks = 0;    // the draw sets: DrawChunks over the dataset's genes
    int n_sets = 1;                   // draw sets over all genes (a shard uses those of the chunks it meets)
    std::vector<int32_t> draws;       // group draws per distinct group size: n_sets blocks of n_boot x size
    std::vector<int64_t> draw_off;    // slot -> offset into draws
    std::vector<int> bslot_D;         // batch slot (distinct composition) -> draws per boot
    std::vector<int32_t> bdraws;      // batch draws (global cell ids) per batch slot: n_sets blocks of n_boot x D
    std::vector<int64_t> bdraw_off;
    std::vector<int> pair_slot, pair_bslot;  // 2 per contrast
    std::vector<int32_t> zi, zi_adj;  // n_zero entries each (1 or N)
    int n_zero = 1;
    const double *batch_models = nullptr;  // when the call's batch.models differ from the dataset's models
    int batch_local_theta = 0, batch_sqlogit = 0;
};

}  // namespace

// one device's part of a dataset: genes [g0, g0 + G)
struct DatasetShard {
    scde_b200_ctx *ctx = nullptr;
    int g0 = 0, G = 0, C = 0, K = 0;
    DiffWorkspace *ws = nullptr;
    ModelSet models, bmodels;
    DBuf<double> mag, prior_y;
    // what the table rows hold: built from `models` (0) or from a call's batch.models (1), for the tcgen05 kernel
    // (fixed-point planes) or the FP64 kernels (FP64 rows)
    int rows_from = 0;
    bool rows_i8 = false;
    DBuf<double> bank, bbank;                 // joint posteriors, [slot][G][ld]
    DBuf<int32_t> cells, draws, bdraws, zi, zi_adj, jflags, gene_set;
    DBuf<int32_t> idx, bidx, aidx;            // [contrast][3][G]
    DBuf<double> z, bz, az;                   // [contrast][G]
    DBuf<RatioContrast> rtab;                 // [pass][contrast] device tables of the batched ratio launches
    StageTimer timer;
    ~DatasetShard() {
        if (ctx) {
            cudaSetDevice(ctx->device);
            ctx->ws_busy = false;
        }
    }
};

struct scde_b200_dataset {
    scde_b200_ctx *owner = nullptr;
    int n_genes = 0, n_cells = 0, n_grid = 0;
    std::vector<DatasetShard *> shards;
    ~scde_b200_dataset() {
        for (auto *s : shards) delete s;
    }
};

namespace {

// rebuild the table rows from the models (from_batch = 0) or from the call's batch.models (1) for the kernel k selects,
// unless they already are
int ensure_rows(DatasetShard &sh, int from_batch, ContractChoice k, StageTimer *tm) {
    scde_b200_ctx *ctx = sh.ctx;
    LpTable &t = sh.ws->table;
    const bool i8 = k.kernel == Contraction::I8;
    if (sh.rows_from == from_batch && sh.rows_i8 == i8 && !from_batch) return SCDE_B200_OK;
    t.want_q = i8;
    sh.rows_from = -1;  // unknown until the rebuild has been queued
    TRY(fill_rows(ctx, t, from_batch ? sh.bmodels : sh.models, sh.mag.p, tm));
    sh.rows_from = from_batch;
    sh.rows_i8 = i8;
    return SCDE_B200_OK;
}

int shard_create(scde_b200_ctx *ctx, const scde_b200_dataset_args *a, int g0, int g1, DatasetShard **out) {
    CHECK_CTX(ctx);
    *out = nullptr;
    TRY(acquire_workspace(ctx));
    DatasetShard *sh = new DatasetShard();
    sh->ctx = ctx;  // from here on, deleting the shard releases the workspace
    sh->ws = ctx->ws;
    const int G = g1 - g0, C = a->n_cells, K = a->n_grid;
    sh->g0 = g0;
    sh->G = G;
    sh->C = C;
    sh->K = K;
    cudaStream_t st = ctx->stream;
    auto body = [&]() -> int {
        SCDE_CUDA(sh->ws->counts.ensure((size_t)G * C));
        SCDE_CUDA(cudaMemcpy2DAsync(sh->ws->counts.p, sizeof(int32_t) * G, a->counts + g0, sizeof(int32_t) * (size_t)a->n_genes,
                                    sizeof(int32_t) * G, C, cudaMemcpyHostToDevice, st));
        TRY(upload_models(sh->models, a->models, C, a->local_theta, a->square_logit_conc, st));
        TRY(upload(sh->prior_y, a->prior_y, (size_t)K, st));
        const std::vector<double> mag = grid_magnitudes(a->prior_x, K);
        TRY(upload(sh->mag, mag.data(), (size_t)K, st));
        LpTable &t = sh->ws->table;
        init_table(ctx, contraction_choice(ctx), t, K, C, sh->models.fast_theta);
        StageTimer &tm = sh->timer;
        tm.reset();
        const int t_all = tm.begin(st);
        TRY(index_from_counts(ctx, t, sh->ws->counts.p, G, 0, G, C, &tm));
        TRY(fill_rows(ctx, t, sh->models, sh->mag.p, &tm));
        tm.end(SCDE_B200_T_TOTAL, t_all, st, 0);
        sh->rows_from = 0;
        sh->rows_i8 = t.want_q;
        SCDE_CUDA(cudaStreamSynchronize(st));
        return SCDE_B200_OK;
    };
    const int r = body();
    if (r != SCDE_B200_OK) {
        cudaStreamSynchronize(st);
        delete sh;
        return r;
    }
    *out = sh;
    return SCDE_B200_OK;
}

int shard_contrasts(DatasetShard &sh, const ContrastPlan &p, const scde_b200_contrast_out *o, scde_b200_stats *stats) {
    scde_b200_ctx *ctx = sh.ctx;
    CHECK_CTX(ctx);
    cudaStream_t st = ctx->stream;
    DiffWorkspace *ws = sh.ws;
    LpTable &t = ws->table;
    StageTimer &tm = sh.timer;
    tm.reset();
    const ContractChoice k = contraction_choice(ctx);
    const int G = sh.G, K = sh.K, nc = p.n_contrasts;
    const int ld = t.ld, nout = 2 * K - 1, ldo = round_up(nout, 8), nadj = 2 * nout - 1, lda = round_up(nadj, 8);
    const int n_slots = (int)p.slot_group.size(), n_bslots = (int)p.bslot_D.size();
    SCDE_CUDA(ws->scr.total.ensure(5));
    SCDE_CUDA(cudaMemsetAsync(ws->scr.total.p, 0, 5 * sizeof(unsigned long long), st));
    const int t_all = tm.begin(st);
    TRY(ensure_rows(sh, 0, k, &tm));
    TRY(upload(sh.cells, p.cells.data(), p.cells.size(), st));
    // this shard's draw sets: those of the chunks it meets.  Only they are uploaded, packed per group size (and per batch
    // composition); sh_draw_off / sh_bdraw_off map a plan offset (the block of all sets) to the packed block on the device.
    const DrawChunks dc = draw_chunks_of(p.N, p.draw_chunks, p.seed, sh.g0, sh.g0 + G);
    std::map<int64_t, int64_t> sh_draw_off;
    std::vector<int64_t> sh_bdraw_off(p.bdraw_off.size());
    {
        auto pack = [&](DBuf<int32_t> &buf, const std::vector<int32_t> &all, const std::vector<std::pair<int64_t, int64_t>> &blocks,
                        std::vector<int64_t> &local) -> int {  // blocks: (plan offset, draws per set)
            int64_t total = 0;
            for (const auto &b : blocks) total += (int64_t)dc.n_sets() * b.second;
            SCDE_CUDA(buf.ensure((size_t)(total > 0 ? total : 1)));
            int64_t off = 0;
            local.clear();
            for (const auto &b : blocks) {
                local.push_back(off);
                const int64_t n = (int64_t)dc.n_sets() * b.second;
                if (n > 0)
                    SCDE_CUDA(cudaMemcpyAsync(buf.p + off, all.data() + b.first + (int64_t)dc.first * b.second,
                                              sizeof(int32_t) * n, cudaMemcpyHostToDevice, st));
                off += n;
            }
            return SCDE_B200_OK;
        };
        std::vector<std::pair<int64_t, int64_t>> blocks;
        for (int s = 0; s < n_slots; ++s)
            if (!sh_draw_off.count(p.draw_off[s])) {
                sh_draw_off[p.draw_off[s]] = -1;
                blocks.emplace_back(p.draw_off[s], (int64_t)p.n_boot * (p.cell_off[s + 1] - p.cell_off[s]));
            }
        std::vector<int64_t> local;
        TRY(pack(sh.draws, p.draws, blocks, local));
        for (size_t i = 0; i < blocks.size(); ++i) sh_draw_off[blocks[i].first] = local[i];
        if (p.has_batch) {
            blocks.clear();
            for (int b = 0; b < n_bslots; ++b) blocks.emplace_back(p.bdraw_off[b], (int64_t)p.n_boot * p.bslot_D[b]);
            TRY(pack(sh.bdraws, p.bdraws, blocks, sh_bdraw_off));
        }
    }
    {
        const std::vector<int32_t> zi = zero_slice(p.zi.data(), p.n_zero, sh.g0, G);
        TRY(upload(sh.zi, zi.data(), zi.size(), st));
        if (p.has_batch) {
            const std::vector<int32_t> za = zero_slice(p.zi_adj.data(), p.n_zero, sh.g0, G);
            TRY(upload(sh.zi_adj, za.data(), za.size(), st));
        }
        SCDE_CUDA(cudaStreamSynchronize(st));  // the host vectors above go out of scope
    }
    if (p.has_batch && p.batch_models)
        TRY(upload_models(sh.bmodels, p.batch_models, sh.C, p.batch_local_theta, p.batch_sqlogit, st));
    const size_t slot_sz = (size_t)G * ld;
    SCDE_CUDA(sh.bank.ensure((size_t)n_slots * slot_sz));
    if (p.has_batch) SCDE_CUDA(sh.bbank.ensure((size_t)n_bslots * slot_sz));
    // tcgen05 status words, one per group joint and per pair of batch joints: a flagged joint is recomputed alone below
    const int n_words = n_slots + (n_bslots + 1) / 2;
    SCDE_CUDA(sh.jflags.ensure((size_t)n_words));
    SCDE_CUDA(cudaMemsetAsync(sh.jflags.p, 0, sizeof(int32_t) * n_words, st));
    if (dc.n_sets() > 1) {
        TRY(upload(sh.gene_set, dc.gene_set.data(), dc.gene_set.size(), st));
        SCDE_CUDA(cudaStreamSynchronize(st));
    }
    const DrawSets sets{dc.n_sets(), dc.n_sets() > 1 ? sh.gene_set.p : nullptr};
    auto group_draws = [&](int s) { return sh.draws.p + sh_draw_off.at(p.draw_off[s]); };
    auto batch_draws = [&](int b) { return sh.bdraws.p + sh_bdraw_off[b]; };
    auto group_joint = [&](int s, ContractChoice kk, bool count) {
        const int n = (int)(p.cell_off[s + 1] - p.cell_off[s]);
        const Joint jt{group_draws(s), n, sh.bank.p + s * slot_sz};
        return run_joint(ctx, kk, t, sh.cells.p + p.cell_off[s], n, &jt, 1, p.n_boot, sets, (double)p.n_boot, ld, ws->scr,
                         sh.jflags.p + s, &tm, count);
    };
    // batch joints b .. b + n - 1 (n <= 2); a pair of joints shares status word n_slots + b / 2
    auto batch_joints = [&](int b, int n, ContractChoice kk, bool count) {
        auto joint = [&](int i) { return Joint{batch_draws(i), p.bslot_D[i], sh.bbank.p + i * slot_sz}; };
        const Joint js[2] = {joint(b), joint(b + n - 1)};
        return run_joint(ctx, kk, t, nullptr, sh.C, js, n, p.n_boot, sets, (double)p.n_boot, ld, ws->scr,
                         sh.jflags.p + n_slots + b / 2, &tm, count);
    };
    for (int s = 0; s < n_slots; ++s) TRY(group_joint(s, k, true));
    if (p.has_batch) {
        if (p.batch_models) TRY(ensure_rows(sh, 1, k, &tm));
        // distinct compositions in pairs: one launch of the tcgen05 kernel for two joints over the same cells and rows
        for (int b = 0; b < n_bslots; b += 2) TRY(batch_joints(b, n_bslots - b < 2 ? 1 : 2, k, true));
    }
    SCDE_CUDA(cudaStreamSynchronize(st));
    std::vector<int32_t> flags(n_words);
    bool any = false;
    TRY(read_status(sh.jflags.p, flags.data(), n_words, &any));
    if (any) {  // only the flagged joints are repeated, on the FP64 kernel (FP64 table rows)
        bool rows = false;
        for (int s = 0; s < n_slots; ++s)
            if (flags[s] & (1 | 4)) {
                if (!rows) TRY(ensure_rows(sh, 0, {Contraction::Tiled}, &tm));
                rows = true;
                TRY(group_joint(s, {Contraction::Tiled}, false));
            }
        rows = false;
        for (int b = 0; b < n_bslots; ++b)
            if (flags[n_slots + b / 2] & (1 | 4)) {
                if (!rows) TRY(ensure_rows(sh, p.batch_models ? 1 : 0, {Contraction::Tiled}, &tm));
                rows = true;
                TRY(batch_joints(b, 1, {Contraction::Tiled}, false));
            }
    }
    // ratio and summary: every contrast in one launch per pass; the 2K-1 posteriors that feed the adjusted pass (or that
    // the caller wants) exist only for a block of contrasts at a time, sized to the free device memory
    const bool keep_post = p.want_post || p.has_batch;
    SCDE_CUDA(sh.idx.ensure((size_t)nc * 3 * G));
    SCDE_CUDA(sh.z.ensure((size_t)nc * G));
    if (p.has_batch) {
        SCDE_CUDA(sh.bidx.ensure((size_t)nc * 3 * G));
        SCDE_CUDA(sh.bz.ensure((size_t)nc * G));
        SCDE_CUDA(sh.aidx.ensure((size_t)nc * 3 * G));
        SCDE_CUDA(sh.az.ensure((size_t)nc * G));
    }
    int nb = nc;
    if (keep_post) {
        const size_t per = sizeof(double) * (size_t)G * ((p.has_batch ? 2 : 1) * (size_t)ldo + (p.want_post && p.has_batch ? lda : 0));
        size_t free_b = 0, total_b = 0;
        SCDE_CUDA(cudaMemGetInfo(&free_b, &total_b));
        const size_t have = sizeof(double) * (ws->post.cap + ws->bpost.cap + ws->apost.cap);
        const size_t fit = (free_b / 2 + have) / per;
        nb = fit < 1 ? 1 : (fit < (size_t)nc ? (int)fit : nc);
        SCDE_CUDA(ws->post.ensure((size_t)nb * G * ldo));
        if (p.has_batch) SCDE_CUDA(ws->bpost.ensure((size_t)nb * G * ldo));
        if (p.has_batch && p.want_post) SCDE_CUDA(ws->apost.ensure((size_t)nb * G * lda));
    }
    const int n_pass = p.has_batch ? 3 : 1;
    std::vector<RatioContrast> tab((size_t)n_pass * nc);
    for (int c = 0; c < nc; ++c) {
        const size_t k = (size_t)(c % nb);
        RatioContrast &m = tab[c];
        m.p1 = sh.bank.p + p.pair_slot[2 * c] * slot_sz;
        m.p2 = sh.bank.p + p.pair_slot[2 * c + 1] * slot_sz;
        m.idx = sh.idx.p + (size_t)c * 3 * G;
        m.z = sh.z.p + (size_t)c * G;
        m.post = keep_post ? ws->post.p + k * G * ldo : nullptr;
        if (!p.has_batch) continue;
        RatioContrast &b = tab[nc + c];
        b.p1 = sh.bbank.p + p.pair_bslot[2 * c] * slot_sz;
        b.p2 = sh.bbank.p + p.pair_bslot[2 * c + 1] * slot_sz;
        b.idx = sh.bidx.p + (size_t)c * 3 * G;
        b.z = sh.bz.p + (size_t)c * G;
        b.post = ws->bpost.p + k * G * ldo;
        RatioContrast &a = tab[2 * nc + c];
        a.p1 = m.post;
        a.p2 = b.post;
        a.idx = sh.aidx.p + (size_t)c * 3 * G;
        a.z = sh.az.p + (size_t)c * G;
        a.post = p.want_post ? ws->apost.p + k * G * lda : nullptr;
    }
    TRY(upload(sh.rtab, tab.data(), tab.size(), st));
    const int64_t N = p.N;
    RatioPasses r = ratio_passes(G, K, ld, sh.prior_y.p, sh.zi.p, sh.zi_adj.p, p.n_zero);
    for (int c0 = 0; c0 < nc; c0 += nb) {
        const int n = nc - c0 < nb ? nc - c0 : nb;
        const int e0 = tm.begin(st);
        r.main.contrasts = sh.rtab.p + c0;
        r.batch.contrasts = sh.rtab.p + nc + c0;
        r.adjusted.contrasts = sh.rtab.p + 2 * nc + c0;
        r.main.n_contrasts = r.batch.n_contrasts = r.adjusted.n_contrasts = n;
        TRY(launch_ratio_passes(r, p.has_batch, st));
        tm.end(SCDE_B200_T_RATIO, e0, st, n_pass);
        for (int c = c0; c < c0 + n && p.want_post; ++c) {
            const size_t k = (size_t)(c - c0);
            if (o->difference_posterior)
                TRY(download_matrix(ctx, ws, G, ws->post.p + k * G * ldo, ldo, nout, o->difference_posterior + (size_t)c * N * nout,
                                    OutPlace{N, sh.g0}));
            if (p.has_batch && o->adjusted_difference_posterior)
                TRY(download_matrix(ctx, ws, G, ws->apost.p + k * G * lda, lda, nadj,
                                    o->adjusted_difference_posterior + (size_t)c * N * nadj, OutPlace{N, sh.g0}));
        }
    }
    tm.end(SCDE_B200_T_TOTAL, t_all, st, 0);
    const OutPlace pl{N, sh.g0};
    for (int c = 0; c < nc; ++c) {
        const size_t i3 = (size_t)c * 3 * G, i1 = (size_t)c * G;
        TRY(download_summary(st, G, sh.idx.p + i3, sh.z.p + i1, o->idx, o->z, pl, c));
        if (!p.has_batch) continue;
        TRY(download_summary(st, G, sh.bidx.p + i3, sh.bz.p + i1, o->batch_idx, o->batch_z, pl, c));
        TRY(download_summary(st, G, sh.aidx.p + i3, sh.az.p + i1, o->adjusted_idx, o->adjusted_z, pl, c));
    }
    if (o->joint_posteriors)
        for (int s = 0; s < n_slots; ++s)
            TRY(download_matrix(ctx, ws, G, sh.bank.p + s * slot_sz, ld, K,
                                o->joint_posteriors + (size_t)p.slot_group[s] * N * K, pl));
    SCDE_CUDA(cudaStreamSynchronize(st));
    return collect_stats(tm, ws, stats);
}

// validation of a contrasts call and everything about it that does not depend on the device
int plan_contrasts(const scde_b200_dataset *ds, const scde_b200_contrast_args *a, const scde_b200_contrast_out *o,
                   ContrastPlan &p) {
    const int C = ds->n_cells, K = ds->n_grid, N = ds->n_genes;
    auto bad = [](const char *fmt, auto... v) {
        set_error(fmt, v...);
        return SCDE_B200_EINVAL;
    };
    if (a->n_groups < 2 || !a->group_offsets || !a->group_cells) return bad("contrasts: need at least two groups");
    if (a->n_contrasts < 1 || !a->pairs) return bad("contrasts: need at least one contrast");
    if (a->n_boot < 1) return bad("contrasts: n_boot must be >= 1");
    TRY(check_draw_chunks(a->draw_chunks, false, "contrasts"));
    if ((o->cz && !o->z) || (o->batch_cz && !o->batch_z) || (o->adjusted_cz && !o->adjusted_z))
        return bad("contrasts: a cZ output needs the matching Z output");
    if (a->group_offsets[0] != 0) return bad("contrasts: group_offsets[0] must be 0");
    for (int g = 0; g < a->n_groups; ++g) {
        const int32_t b = a->group_offsets[g], e = a->group_offsets[g + 1];
        if (e <= b) return bad("contrasts: group %d is empty", g);
        for (int32_t i = b; i < e; ++i) {
            const int32_t c = a->group_cells[i];
            if (c < 0 || c >= C) return bad("contrasts: group %d: cell %d outside [0, %d)", g, c, C);
            if (i > b && c <= a->group_cells[i - 1]) return bad("contrasts: group %d: cell ids not ascending at %d", g, c);
        }
    }
    p.has_batch = a->batch != nullptr && a->n_batch_levels > 1;
    if (a->n_zero != 1 && a->n_zero != N) return bad("contrasts: n_zero must be 1 or n_genes");
    if (!a->zero_index || (p.has_batch && !a->zero_index_adjusted))
        return bad("contrasts: zero_index (and zero_index_adjusted with batch) are required");
    TRY(validate_index(a->zero_index, (size_t)a->n_zero, 1, 2 * K, "zero_index"));
    p.zi.assign(a->zero_index, a->zero_index + a->n_zero);
    BatchPools bp;  // the draw pools of the batch joints below
    if (p.has_batch) {
        TRY(validate_index(a->zero_index_adjusted, (size_t)a->n_zero, 1, 4 * K - 2, "zero_index_adjusted"));
        p.zi_adj.assign(a->zero_index_adjusted, a->zero_index_adjusted + a->n_zero);
        TRY(batch_pools(a->batch, C, a->n_batch_levels, bp));
    }
    p.C = C;
    p.K = K;
    p.N = N;
    p.n_zero = a->n_zero;
    p.n_contrasts = a->n_contrasts;
    p.n_boot = a->n_boot;
    p.seed = a->seed;
    p.draw_chunks = a->draw_chunks;
    const std::vector<int32_t> seeds = chunk_seeds(N, a->draw_chunks, a->seed);
    p.n_sets = (int)seeds.size();
    p.want_post = o->difference_posterior || o->adjusted_difference_posterior;
    std::vector<int> slot_of(a->n_groups, -1);
    p.pair_slot.resize(2 * (size_t)a->n_contrasts);
    for (int c = 0; c < a->n_contrasts; ++c) {
        const int ga = a->pairs[2 * c], gb = a->pairs[2 * c + 1];
        if (ga < 0 || ga >= a->n_groups || gb < 0 || gb >= a->n_groups)
            return bad("contrast %d names group %d outside [0, %d)", c, ga < 0 || ga >= a->n_groups ? ga : gb, a->n_groups);
        if (ga == gb) return bad("contrast %d compares group %d with itself", c, ga);
        // the two sides of one contrast must not share a cell (both lists are ascending)
        int32_t i = a->group_offsets[ga], j = a->group_offsets[gb];
        while (i < a->group_offsets[ga + 1] && j < a->group_offsets[gb + 1]) {
            const int32_t x = a->group_cells[i], y = a->group_cells[j];
            if (x == y) return bad("contrast %d: groups %d and %d share cell %d", c, ga, gb, x);
            if (x < y) ++i; else ++j;
        }
        for (int s = 0; s < 2; ++s) {
            const int g = s ? gb : ga;
            if (slot_of[g] < 0) {
                slot_of[g] = (int)p.slot_group.size();
                p.slot_group.push_back(g);
            }
            p.pair_slot[2 * c + s] = slot_of[g];
        }
    }
    // group joints: cells of every slot, draws once per distinct group size (local indices, src/jpmatLogBoot.cpp:221,254-257)
    // and draw set; the draws are generated below, on parallel host threads, one (size or composition, set) each
    const int S = p.n_sets;
    std::vector<std::pair<int64_t, int>> group_tasks;  // (offset of the set's block, size)
    std::map<int, int64_t> draws_of_size;
    p.cell_off.assign(1, 0);
    for (int g : p.slot_group) {
        const int32_t b = a->group_offsets[g], e = a->group_offsets[g + 1];
        p.cells.insert(p.cells.end(), a->group_cells + b, a->group_cells + e);
        p.cell_off.push_back((int64_t)p.cells.size());
        const int n = e - b;
        auto it = draws_of_size.find(n);
        if (it == draws_of_size.end()) {
            it = draws_of_size.emplace(n, (int64_t)p.draws.size()).first;
            for (int s = 0; s < S; ++s) group_tasks.emplace_back(it->second + (int64_t)s * a->n_boot * n, n);
            p.draws.resize(p.draws.size() + (size_t)S * a->n_boot * n);
        }
        p.draw_off.push_back(it->second);
    }
    TRY(parallel_for((int)group_tasks.size(), [&](int i) -> int {
        const auto &tk = group_tasks[i];
        return scde_b200_boot_indices(seeds[(size_t)i % S], tk.second, a->n_boot, p.draws.data() + tk.first);
    }));
    if (!p.has_batch) return SCDE_B200_OK;
    // batch joints: one per distinct composition table(batch[group]) (R/functions.R:355-357)
    const int L = a->n_batch_levels;
    std::map<std::vector<int32_t>, int> bslot_of;
    std::vector<std::vector<int32_t>> bcomp;  // composition of every batch slot
    std::vector<int> bslot_of_slot(p.slot_group.size());
    for (size_t s = 0; s < p.slot_group.size(); ++s) {
        std::vector<int32_t> comp;
        const int D = batch_composition(a->batch, L, p.cells.data() + p.cell_off[s], (size_t)(p.cell_off[s + 1] - p.cell_off[s]),
                                        comp);
        auto it = bslot_of.find(comp);
        if (it == bslot_of.end()) {
            it = bslot_of.emplace(comp, (int)p.bslot_D.size()).first;
            p.bslot_D.push_back(D);
            p.bdraw_off.push_back((int64_t)p.bdraws.size());
            p.bdraws.resize(p.bdraws.size() + (size_t)S * a->n_boot * D);
            bcomp.push_back(comp);
        }
        bslot_of_slot[s] = it->second;
    }
    TRY(parallel_for((int)bcomp.size() * S, [&](int i) -> int {
        const int b = i / S, set = i % S;
        return scde_b200_batch_boot_indices(seeds[set], L, bp.off.data(), bp.pool.data(), bcomp[b].data(), a->n_boot,
                                            p.bdraws.data() + p.bdraw_off[b] + (int64_t)set * a->n_boot * p.bslot_D[b]);
    }));
    p.pair_bslot.resize(p.pair_slot.size());
    for (size_t i = 0; i < p.pair_slot.size(); ++i) p.pair_bslot[i] = bslot_of_slot[p.pair_slot[i]];
    if (a->batch_models) {
        p.batch_models = a->batch_models;
        p.batch_local_theta = a->batch_local_theta;
        p.batch_sqlogit = a->batch_square_logit_conc;
    }
    return SCDE_B200_OK;
}

}  // namespace

extern "C" {

int scde_b200_dataset_create(scde_b200_ctx *ctx, const scde_b200_dataset_args *a, scde_b200_dataset **out,
                             scde_b200_stats *stats) {
    CHECK_CTX(ctx);
    if (!a || !out) {
        set_error("dataset_create: null argument");
        return SCDE_B200_EINVAL;
    }
    *out = nullptr;
    if (!a->counts || !a->models || !a->prior_x || !a->prior_y || a->n_genes < 1 || a->n_cells < 1 || a->n_grid < 2) {
        set_error("dataset_create: bad arguments");
        return SCDE_B200_EINVAL;
    }
    const std::vector<scde_b200_ctx *> devs = context_devices(ctx);
    for (auto *d : devs) TRY(workspace_busy(d));
    const int n = (int)devs.size() < a->n_genes ? (int)devs.size() : a->n_genes;
    scde_b200_dataset *ds = new scde_b200_dataset();
    ds->owner = ctx;
    ds->n_genes = a->n_genes;
    ds->n_cells = a->n_cells;
    ds->n_grid = a->n_grid;
    ds->shards.assign(n, nullptr);
    std::vector<scde_b200_stats> sst(n);
    const int r = on_shards(n, devs, [&](int i) -> int {
        int b = 0, e = 0;
        shard_range(a->n_genes, n, i, &b, &e);
        TRY(shard_create(devs[i], a, b, e, &ds->shards[i]));
        ds->shards[i]->timer.collect(&sst[i]);
        sst[i].table_rows = ds->shards[i]->ws->table.n_rows;
        return SCDE_B200_OK;
    }, &sst, stats);
    if (r != SCDE_B200_OK) {
        for (auto *&s : ds->shards) {
            delete s;
            s = nullptr;
        }
        delete ds;
        cudaSetDevice(ctx->device);
        return r;
    }
    *out = ds;
    return SCDE_B200_OK;
}

int scde_b200_dataset_contrasts(scde_b200_ctx *ctx, scde_b200_dataset *ds, const scde_b200_contrast_args *a,
                                const scde_b200_contrast_out *o, scde_b200_stats *stats) {
    CHECK_CTX(ctx);
    if (!ds || !a || !o) {
        set_error("dataset_contrasts: null argument");
        return SCDE_B200_EINVAL;
    }
    if (ds->owner != ctx) {
        set_error("dataset_contrasts: the dataset belongs to another context");
        return SCDE_B200_EINVAL;
    }
    ContrastPlan p;
    try {
        TRY(plan_contrasts(ds, a, o, p));
    } catch (const std::bad_alloc &) {
        set_error("dataset_contrasts: host allocation failed");
        return SCDE_B200_ENOMEM;
    }
    const std::vector<scde_b200_ctx *> devs = context_devices(ctx);
    const int n = (int)ds->shards.size();
    std::vector<scde_b200_stats> sst(n);
    TRY(on_shards(n, devs, [&](int i) -> int { return shard_contrasts(*ds->shards[i], p, o, &sst[i]); }, &sst, stats));
    // Benjamini-Hochberg per contrast over all genes, on the host, once every shard has landed
    for (int c = 0; c < a->n_contrasts; ++c) bh_outputs(o, p.has_batch, ds->n_genes, c);
    return SCDE_B200_OK;
}

void scde_b200_dataset_free(scde_b200_ctx *ctx, scde_b200_dataset *ds) {
    delete ds;  // every shard releases its context's workspace
    if (ctx) cudaSetDevice(ctx->device);
}

}  // extern "C"
