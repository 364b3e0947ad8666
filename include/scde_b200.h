/*
 * scde_b200.h -- C ABI of libscde_b200.so: the B200 (sm_100a) implementation of scde's
 * differential-expression posterior hot path.
 *
 * The entry points are what the reference's R layer would bind in place of its native
 * `.Call(..., PACKAGE = "scde")` sites (reference paths are relative to the scde source tree):
 *
 *   scde_b200_log_boot_posterior        <- .Call("logBootPosterior", ...)       R/functions.R:613,637
 *                                          (RcppExport at src/jpmatLogBoot.cpp:100)
 *   scde_b200_log_boot_batch_posterior  <- .Call("logBootBatchPosterior", ...)  R/functions.R:611,635
 *                                          (src/jpmatLogBoot.cpp:343)
 *   scde_b200_mat_slide_mult            <- .Call("matSlideMult", ...)           R/functions.R:3545
 *                                          (src/matSlideMult.cpp:5)
 *   scde_b200_jpmat_log_boot            <- .Call("jpmatLogBoot", ...)           R/functions.R:3535
 *   scde_b200_jpmat_log_batch_boot      <- .Call("jpmatLogBatchBoot", ...)      R/functions.R:3541
 *   scde_b200_ratio_posterior_summary   <- calculate.ratio.posterior + quick.distribution.summary
 *                                          (R/functions.R:3491-3531, 5039-5053) fused on the device
 *   scde_b200_expression_difference     <- the whole of scde.expression.difference's numeric work
 *                                          (R/functions.R:304-408) with jp kept in HBM
 *   scde_b200_expression_magnitude      <- scde.expression.magnitude (R/functions.R:694-697)
 *
 * Conventions
 *   - plain pointers and sizes only; every matrix is column-major (R layout): element (i, j) of an
 *     r x c matrix is at [i + r * j];
 *   - all buffers are caller-owned HOST memory unless a name ends in `_dev`; outputs are written into
 *     caller-allocated buffers; the library owns only device memory and frees it before returning
 *     (or keeps it in an explicit handle);
 *   - every function returns 0 on success, a negative SCDE_B200_E* code otherwise, never throws and
 *     never longjmps; scde_b200_last_error() describes the last failure on the calling thread;
 *   - there is NO CPU fallback: without a usable CUDA device every compute entry point fails with
 *     SCDE_B200_ENODEVICE;
 *   - calls on one context are synchronous with respect to the host and must not be issued from a
 *     forked child of a process that already created a CUDA context (R's mclapply/papply).
 */
#ifndef SCDE_B200_H
#define SCDE_B200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define SCDE_B200_VERSION 100

#if defined(__GNUC__)
#define SCDE_B200_API __attribute__((visibility("default")))
#else
#define SCDE_B200_API
#endif

enum {
    SCDE_B200_OK = 0,
    SCDE_B200_EINVAL = -1,    /* bad argument (shape, index out of range, NULL) */
    SCDE_B200_ENODEVICE = -2, /* no CUDA device / driver */
    SCDE_B200_ECUDA = -3,     /* CUDA runtime error (message in last_error) */
    SCDE_B200_ENOMEM = -4,    /* device or host allocation failed */
    SCDE_B200_ELIMIT = -5     /* a documented capacity limit was exceeded */
};

/* Column order of the 12-column model matrix (R/functions.R:601; src/jpmatLogBoot.cpp:101-112).
 * Columns a model family does not have may hold NaN/NA. */
enum {
    SCDE_B200_CONC_B = 0, SCDE_B200_CONC_A, SCDE_B200_FAIL_R, SCDE_B200_CORR_B, SCDE_B200_CORR_A,
    SCDE_B200_CORR_THETA, SCDE_B200_CORR_LTHETA_B, SCDE_B200_CORR_LTHETA_T, SCDE_B200_CORR_LTHETA_M,
    SCDE_B200_CORR_LTHETA_S, SCDE_B200_CORR_LTHETA_R, SCDE_B200_CONC_A2, SCDE_B200_N_MODEL_COLS
};

typedef struct scde_b200_ctx scde_b200_ctx;

/* ---- context ------------------------------------------------------------------------------- */
SCDE_B200_API int scde_b200_version(void);
SCDE_B200_API const char *scde_b200_last_error(void);
/* number of visible CUDA devices (0 when there is no driver); never fails */
SCDE_B200_API int scde_b200_device_count(void);
/* create a context on CUDA device `device` with its own non-blocking stream */
SCDE_B200_API int scde_b200_create(int device, scde_b200_ctx **out);
SCDE_B200_API void scde_b200_destroy(scde_b200_ctx *ctx);
/* the context's cudaStream_t (as void*), so callers can record their own events on it */
SCDE_B200_API void *scde_b200_stream(scde_b200_ctx *ctx);
/* blocks until all work queued on the context's stream has finished */
SCDE_B200_API int scde_b200_synchronize(scde_b200_ctx *ctx);

/*
 * A context over several CUDA devices of one node.  scde_b200_expression_difference on such a context shards the genes
 * into contiguous ranges, one per device, runs every shard on its own host thread, and the shards' results land in the
 * caller's buffers by device-to-host copies -- no inter-GPU traffic.  The number of devices does not change results: the
 * draws follow the call's `seed` and `draw_chunks` (the reference's n.cores, see scde_b200_diff_args) whatever the
 * sharding.  devices == NULL: devices 0 .. n_devices-1.  Every other entry point uses the first device of the list.
 */
SCDE_B200_API int scde_b200_create_multi(int n_devices, const int *devices, scde_b200_ctx **out);
/* number of devices of the context (1 for scde_b200_create) */
SCDE_B200_API int scde_b200_n_devices(const scde_b200_ctx *ctx);

/*
 * Behavioural switches of a context (SURVEY.md section 5: the reference has function arguments only -- no global
 * options, no environment variables -- so neither has the library).  scde_b200_get_options fills the defaults (or the
 * current values); scde_b200_set_options applies to every later call on the context (and on its per-device children).
 */
typedef struct {
    int32_t contract_kernel;    /* 0 auto (tcgen05 fixed point where it applies), 1 generic FP64, 2 tiled FP64 (DMMA), 3 tcgen05 */
    int32_t zero_base;          /* 1: rows hold lp(x) - lp(0), the contraction visits non-zero counts only */
    int32_t fused_fixed_point;  /* 1: the row kernel emits the fixed-point planes itself (FP64 rows of non-zero counts not stored) */
    int32_t lp_rows_kernel;     /* 0: register-resident row kernel (default); 1: the per-element kernel it replaced (tests) */
    int32_t count_chunks;       /* one-shot call: the count matrix goes up in this many cell chunks (default 8, 1..64) */
    int32_t split_front;        /* 1: the first group's joint runs under the upload of the second group's cells */
    int32_t uniform_chunks;     /* 1: equal chunks instead of a small first and last one */
    int32_t pipeline_front;     /* 1: chunks are processed as they land; 0: wait for the whole matrix */
    int32_t item_order;         /* tcgen05 contraction: 0 = the pieces of a gene on neighbouring SMs, 1 = piece-major (default) */
    int32_t hot_rank;           /* table rows whose rank within their cell is <= hot_rank are loaded with the L2 evict_last
                                   policy; < 0: no cache hints */
    int32_t cold_evict_first;   /* with hot_rank >= 0: the other rows are loaded evict_first (1) or without a priority (0) */
    int32_t trace;              /* 1: host wall-clock of the phases of the one-shot call on stderr */
    int32_t epilogue_timing;    /* 1: cycle counters of the tcgen05 kernel's epilogue on stderr */
    int32_t debug_contract;     /* FP64 tiled kernel: diagnostic mode (0 = off) */
    int32_t ring_stages;        /* tcgen05 contraction: stages of the shared-memory ring, 0 = default (10); 7 or 8 (experiments) */
    int32_t twin_batch_joints;  /* 1 (default): two contractions over the same cells and rows share the launches of the tcgen05
                                   kernel (paired items on neighbouring SMs): the two composition-sampled joints of a
                                   batch-corrected call, and the two passes of more than 104 randomizations */
    int32_t prune_pieces;       /* 1 (default): the tcgen05 contraction skips the (gene, piece) items whose grid points bounds
                                   computed before it prove invisible to the soft-max (DESIGN.md 4.3); results are unchanged */
    int32_t reserved[4];
} scde_b200_options;
SCDE_B200_API int scde_b200_get_options(const scde_b200_ctx *ctx, scde_b200_options *opt);
SCDE_B200_API int scde_b200_set_options(scde_b200_ctx *ctx, const scde_b200_options *opt);

/* ---- bootstrap draws (host; glibc TYPE_3 additive-feedback rand() restated) ---------------- */
/* Reproduces `srand(seed); for b<n_boot, j<n: while(n <= (rj = rand()/(RAND_MAX/n)));`
 * (src/jpmatLogBoot.cpp:221,254-257) without touching libc's global state.  out[b*n + j], draw order. */
SCDE_B200_API int scde_b200_boot_indices(int32_t seed, int32_t n, int32_t n_boot, int32_t *out);
/* Batch variant (src/jpmatLogBoot.cpp:467-481): per boot, for each level k with composition[k] > 0,
 * composition[k] draws from pool k = pool_cells[pool_offsets[k] .. pool_offsets[k+1]); the value stored is
 * the global cell id.  out[b*D + d], D = sum of positive composition entries. */
SCDE_B200_API int scde_b200_batch_boot_indices(int32_t seed, int32_t n_levels, const int32_t *pool_offsets,
                                 const int32_t *pool_cells, const int32_t *composition, int32_t n_boot,
                                 int32_t *out);

/* ---- joint posteriors ---------------------------------------------------------------------- */
/*
 * logBootPosterior.  Arguments mirror the .Call site:
 *   models[n_cells*12]; ucl_flat / ucl_offsets[n_cells+1] = the list `ucl` flattened; uci[n_genes*n_cells]
 *   0-based indices into ucl[[cell]]; magnitudes[n_grid] natural-log grid (may contain -Inf);
 *   n_boot, seed; return_individual 0..3; local_theta, square_logit_conc, ensemble flags.
 *   boot_idx: optional explicit draws [n_boot*n_cells] (NULL = generate from `seed`).
 * Outputs: jp[n_genes*n_grid]; modes[n_genes*n_cells] (return_individual 1|3, else may be NULL);
 *   post[n_cells * n_genes*n_grid] = the list of per-cell matrices back to back (2|3, else NULL).
 */
SCDE_B200_API int scde_b200_log_boot_posterior(scde_b200_ctx *ctx, const double *models, int32_t n_cells,
                                 const int32_t *ucl_flat, const int32_t *ucl_offsets, const int32_t *uci,
                                 int32_t n_genes, const double *magnitudes, int32_t n_grid, int32_t n_boot,
                                 int32_t seed, const int32_t *boot_idx, int32_t return_individual,
                                 int32_t local_theta, int32_t square_logit_conc, int32_t ensemble, double *jp,
                                 double *modes, double *post);

/*
 * logBootBatchPosterior: as above plus BatchIL (flattened: batchil_offsets[n_levels+1], batchil_cells) and
 * Composition[n_levels].  boot_idx: optional [n_boot*D] global cell ids.  As in the reference, `modes`
 * is produced for return_individual == 1 only and 3 behaves like 2.
 */
SCDE_B200_API int scde_b200_log_boot_batch_posterior(scde_b200_ctx *ctx, const double *models, int32_t n_cells,
                                       const int32_t *ucl_flat, const int32_t *ucl_offsets, const int32_t *uci,
                                       int32_t n_genes, const double *magnitudes, int32_t n_grid,
                                       int32_t n_levels, const int32_t *batchil_offsets,
                                       const int32_t *batchil_cells, const int32_t *composition, int32_t n_boot,
                                       int32_t seed, const int32_t *boot_idx, int32_t return_individual,
                                       int32_t local_theta, int32_t square_logit_conc, double *jp, double *modes,
                                       double *post);

/* Legacy dense form: matl = n_mat matrices (n_rows x n_cols, column-major) back to back.  Not divided by
 * n_boot, exactly as the reference (the R caller renormalises, R/functions.R:3464-3465). */
SCDE_B200_API int scde_b200_jpmat_log_boot(scde_b200_ctx *ctx, const double *matl, int32_t n_mat, int32_t n_rows,
                             int32_t n_cols, int32_t n_boot, int32_t seed, const int32_t *boot_idx, double *jp);
/* matl holds all pools' matrices back to back; pool k = matrices pool_offsets[k] .. pool_offsets[k+1]. */
SCDE_B200_API int scde_b200_jpmat_log_batch_boot(scde_b200_ctx *ctx, const double *matl, int32_t n_levels,
                                   const int32_t *pool_offsets, const int32_t *composition, int32_t n_rows,
                                   int32_t n_cols, int32_t n_boot, int32_t seed, const int32_t *boot_idx,
                                   double *jp);

/* ---- group-difference posterior ------------------------------------------------------------ */
/* matSlideMult: m1, m2 n_rows x n  ->  out n_rows x (2n-1); multiply and add are rounded separately in
 * ascending j, so the result is bit-identical to the reference's loop on an x86-64 build without FMA. */
SCDE_B200_API int scde_b200_mat_slide_mult(scde_b200_ctx *ctx, const double *m1, const double *m2, int32_t n_rows, int32_t n,
                             double *out);

/*
 * calculate.ratio.posterior fused with quick.distribution.summary's per-gene part.
 *   pmat1, pmat2: n_genes x n; prior_y[n] or NULL (skip.prior.adjustment = TRUE);
 *   zero_index: 1-based grid position of the H0 value per gene (n_zero == n_genes) or shared (n_zero == 1)
 *     -- what get.ratio.posterior.Z.score calls `zi` (R/functions.R:3519,3524).
 * Outputs: idx[n_genes*3] 0-based grid indices (lb, mle, ub); z[n_genes];
 *   posterior (optional, may be NULL): n_genes x (2n-1) normalised ratio posterior.
 * The fold-change values, ce and cZ are host work on these (see scde_b200_bh_cz).
 */
SCDE_B200_API int scde_b200_ratio_posterior_summary(scde_b200_ctx *ctx, const double *pmat1, const double *pmat2,
                                      int32_t n_genes, int32_t n, const double *prior_y,
                                      const int32_t *zero_index, int32_t n_zero, int32_t *idx, double *z,
                                      double *posterior);

/* cZ = sign(Z) * qnorm(p.adjust(pnorm(|Z|, lower = F), "BH"), lower = F)  (R/functions.R:5051); host. */
SCDE_B200_API int scde_b200_bh_cz(const double *z, int32_t n, double *cz);

/* ---- whole differential-expression call ---------------------------------------------------- */
typedef struct {
    int32_t n_genes, n_cells, n_grid;
    const int32_t *counts;   /* n_genes x n_cells raw counts, cells ordered as the model rows */
    const double *models;    /* n_cells x 12 (corr.a already clamped to >= 1e-10 by the caller) */
    const double *prior_x;   /* n_grid: prior$x (log10(FPM+1) grid) */
    const double *prior_y;   /* n_grid: prior$y */
    const int32_t *group;    /* n_cells: 0 = first factor level, 1 = second, <0 = NA (ignored) */
    const int32_t *batch;    /* n_cells batch level codes 0..n_batch_levels-1 (< 0 = NA: in no pool, not in the
                                composition, as tapply / table drop NA), or NULL (no correction) */
    int32_t n_batch_levels;
    int32_t n_boot;          /* n.randomizations */
    int32_t seed;            /* Seed handed to srand(); 1 reproduces the reference (see draw_chunks for its n.cores) */
    /* optional explicit draws; NULL = generate from `seed`.  [0],[1]: group joints (local indices into the
     * group's cells, n_boot x |group|); [2],[3]: batch joints (global cell ids, n_boot x number of the group's cells with
     * a non-NA batch). */
    const int32_t *boot_idx[4];
    const int32_t *zero_index; /* 1-based H0 grid position(s) on the 2K-1 fold-change grid */
    int32_t n_zero;            /* 1 or n_genes */
    const int32_t *zero_index_adjusted; /* same on the 4K-3 batch-adjusted grid (batch only) */
    int32_t local_theta, square_logit_conc;
    int32_t gene_begin, gene_end; /* process genes [gene_begin, gene_end) of `counts` (0,0 = all): the
                                     multi-GPU gene shard; outputs are indexed from gene_begin */
    /* batch.models (R/functions.R:304,356): the error models of the two composition-sampled joints, n_cells x 12, rows in
     * the order of `models`; NULL = the same models (the reference's default).  With their own column-presence flags. */
    const double *batch_models;
    int32_t batch_local_theta, batch_square_logit_conc;
    /* The reference's n.cores (R/functions.R:606-617): scde.posteriors splits the genes into n contiguous chunks and
     * draws every chunk's randomizations with Seed = the chunk's first gene (1-based).  With n = draw_chunks > 1 and
     * n_genes > n, chunk i is genes [b_i, e_i) of shard_range(n_genes, n, i) (the first n_genes % n chunks one gene
     * longer) and its draws -- of every joint, group and batch -- come from seed + b_i; otherwise one draw set from
     * `seed` for all genes.  0 or 1: one draw set (n.cores = 1).  Chunks are over the call's n_genes, not its gene range
     * or device shard.  < 0, or > 1 together with an explicit boot_idx: SCDE_B200_EINVAL; above
     * SCDE_B200_MAX_DRAW_CHUNKS: SCDE_B200_ELIMIT. */
    int32_t draw_chunks;
} scde_b200_diff_args;
/* the largest draw_chunks: it bounds the per-set W and Z memory and the number of host threads generating draws */
#define SCDE_B200_MAX_DRAW_CHUNKS 256

typedef struct {
    /* per processed gene; any pointer may be NULL to skip that output */
    int32_t *idx;            /* n x 3 (lb, mle, ub) 0-based on the 2K-1 grid */
    double *z;               /* n */
    int32_t *batch_idx;      /* batch.effect summary, n x 3 */
    double *batch_z;
    int32_t *adjusted_idx;   /* batch.adjusted summary on the 4K-3 grid, n x 3 */
    double *adjusted_z;
    double *difference_posterior;          /* n x (2K-1) */
    double *batch_difference_posterior;    /* n x (2K-1) */
    double *adjusted_difference_posterior; /* n x (4K-3) */
    double *joint_posteriors[2];           /* n x K each */
    double *batch_joint_posteriors[2];     /* n x K each */
    /* cZ = sign(Z) qnorm(p.adjust(pnorm(|Z|, lower = F), "BH"), lower = F) (R/functions.R:5051) of the matching Z output, n
     * each; computed on the host over the genes THIS call processes -- the reference's cZ when that is every gene (with a
     * gene range the caller gathers Z and uses scde_b200_bh_cz).  Filled by scde_b200_expression_difference only. */
    double *cz, *batch_cz, *adjusted_cz;
} scde_b200_diff_out;

/* Per-stage device timings of the last run on a job, in milliseconds (CUDA events on the context stream),
 * and the number of kernel launches.  Index with SCDE_B200_T_*. */
enum {
    SCDE_B200_T_DEDUP = 0,   /* unique-count table indices */
    SCDE_B200_T_LPTABLE,     /* per-cell log-posterior rows */
    SCDE_B200_T_CONTRACT,    /* bootstrap contraction (all joints); the FP64 kernels' time includes their soft-max */
    SCDE_B200_T_RATIO,       /* sliding product + summary (all passes) */
    SCDE_B200_T_OTHER,       /* W build, entry lists, zero-count base sums, memsets */
    SCDE_B200_T_SOFTMAX,     /* soft-max over the grid + average over boots after the tcgen05 contraction kernel */
    SCDE_B200_T_BOUND,       /* pruning before the tcgen05 contraction: bound pass, live-item decision and list */
    SCDE_B200_T_TOTAL,
    SCDE_B200_T_COUNT
};
typedef struct {
    float ms[SCDE_B200_T_COUNT];
    int32_t launches[SCDE_B200_T_COUNT];
    int64_t table_rows;      /* rows in the log-posterior table */
    int64_t contract_cells;  /* list entries (gene x cell pairs) the contraction visited, summed over all joints */
    int64_t prune_items;     /* (gene, piece) items of the pruned tcgen05 launches, summed over joints and passes (a twin
                                launch counts its pairs once) */
    int64_t prune_live;      /* ... of which were contracted */
    int64_t prune_work;      /* the same items weighted by their gene's list length: (visited pair, piece) units, i.e. the
                                gather the launches would have done unpruned */
    int64_t prune_live_work; /* ... of which were gathered */
} scde_b200_stats;

/* One-shot: host buffers in, host buffers out (uploads, runs, downloads).  The count matrix goes up in cell chunks that are
 * processed as they land; when the cells of group 0 lead the matrix (cells ordered by group) that group's joint
 * posterior is computed while the rest is still uploading.  Any cell order gives the same results. */
SCDE_B200_API int scde_b200_expression_difference(scde_b200_ctx *ctx, const scde_b200_diff_args *args,
                                    const scde_b200_diff_out *out, scde_b200_stats *stats);

/* Split form for device-resident timing: upload once, run any number of times, download. */
typedef struct scde_b200_diff_job scde_b200_diff_job;
SCDE_B200_API int scde_b200_diff_upload(scde_b200_ctx *ctx, const scde_b200_diff_args *args, int32_t want_posteriors,
                          scde_b200_diff_job **job);
/* queues all device work on the context stream and returns without waiting for it */
SCDE_B200_API int scde_b200_diff_run(scde_b200_ctx *ctx, scde_b200_diff_job *job);
/* waits for the stream, then copies results to the host buffers in `out`; fills `stats` if not NULL */
SCDE_B200_API int scde_b200_diff_download(scde_b200_ctx *ctx, scde_b200_diff_job *job, const scde_b200_diff_out *out,
                            scde_b200_stats *stats);
SCDE_B200_API void scde_b200_diff_free(scde_b200_ctx *ctx, scde_b200_diff_job *job);

/* ---- many contrasts on one resident dataset ------------------------------------------------- */
/*
 * A dataset holds the count matrix, its unique-count index and the log-posterior table of ALL its cells on the device, so
 * that any number of two-group contrasts over those cells can be computed without rebuilding them.  Every contrast (A, B)
 * returns bit for bit what scde_b200_expression_difference returns for the same data, options, n_boot, seed, expectation
 * and batch, with group code 0 on A's cells, 1 on B's cells and -1 on every other cell -- except where the tcgen05
 * contraction had to fall back to the FP64 kernel (see DESIGN.md, "Many contrasts"): there the affected contrasts agree
 * with the one-shot call within the oracle tolerances.
 *
 * Each group's joint posterior is computed once per call however many contrasts name it (the draws of a group depend on
 * the seed, n_boot, draw_chunks and the group's size only), and each distinct batch composition's joint once.
 *
 * A dataset holds its context's differential-expression workspace until scde_b200_dataset_free: while it is alive,
 * scde_b200_expression_difference, scde_b200_diff_upload and a second scde_b200_dataset_create on that context fail with
 * SCDE_B200_EINVAL ("another expression_difference job is alive").  On a scde_b200_create_multi context the dataset is one
 * per-device dataset per contiguous gene range (the split of scde_b200_expression_difference).
 */
typedef struct {
    int32_t n_genes, n_cells, n_grid;
    const int32_t *counts;   /* n_genes x n_cells raw counts, cells ordered as the model rows */
    const double *models;    /* n_cells x 12 (corr.a already clamped to >= 1e-10 by the caller) */
    const double *prior_x;   /* n_grid */
    const double *prior_y;   /* n_grid */
    int32_t local_theta, square_logit_conc;
} scde_b200_dataset_args;

typedef struct {
    /* groups as flattened cell lists: group i = group_cells[group_offsets[i] .. group_offsets[i+1]), model-row ids in
     * ascending order, at least one cell each.  Groups may share cells, except the two groups of one contrast. */
    int32_t n_groups;
    const int32_t *group_offsets;  /* n_groups + 1 */
    const int32_t *group_cells;
    int32_t n_contrasts;
    const int32_t *pairs;          /* 2 * n_contrasts group ids: contrast c is (pairs[2c], pairs[2c+1]) = (A, B) */
    int32_t n_boot, seed;
    const int32_t *zero_index;     /* as in scde_b200_diff_args, shared by every contrast */
    int32_t n_zero;
    const int32_t *zero_index_adjusted;
    const int32_t *batch;          /* n_cells batch level codes (< 0 = NA) or NULL */
    int32_t n_batch_levels;
    const double *batch_models;    /* n_cells x 12 or NULL (= models), with their own column-presence flags */
    int32_t batch_local_theta, batch_square_logit_conc;
    int32_t draw_chunks;           /* as in scde_b200_diff_args, over the dataset's n_genes */
} scde_b200_contrast_args;

/* Outputs, any pointer may be NULL.  Per-contrast blocks back to back: contrast c's block of a G x m output starts at
 * c * G * m (G = the dataset's genes) and is column-major like the matching scde_b200_diff_out field.  cz, batch_cz and
 * adjusted_cz are Benjamini-Hochberg over all genes of the contrast and need the matching z output. */
typedef struct {
    int32_t *idx;            /* n_contrasts x (G x 3) */
    double *z, *cz;          /* n_contrasts x G */
    int32_t *batch_idx;
    double *batch_z, *batch_cz;
    int32_t *adjusted_idx;
    double *adjusted_z, *adjusted_cz;
    double *difference_posterior;          /* n_contrasts x (G x (2K-1)) */
    double *adjusted_difference_posterior; /* n_contrasts x (G x (4K-3)), batch only */
    double *joint_posteriors;              /* n_groups x (G x K); groups that no contrast names are left untouched */
} scde_b200_contrast_out;

typedef struct scde_b200_dataset scde_b200_dataset;
/* uploads the counts, builds the index and the table; stats (may be NULL) report the dedup and table stages */
SCDE_B200_API int scde_b200_dataset_create(scde_b200_ctx *ctx, const scde_b200_dataset_args *args, scde_b200_dataset **out,
                                           scde_b200_stats *stats);
/* every contrast of `args` in one call; stats (may be NULL): launches[CONTRACT] and contract_cells count one contraction
 * per distinct group and one per pair of batch joints */
SCDE_B200_API int scde_b200_dataset_contrasts(scde_b200_ctx *ctx, scde_b200_dataset *ds, const scde_b200_contrast_args *args,
                                              const scde_b200_contrast_out *out, scde_b200_stats *stats);
SCDE_B200_API void scde_b200_dataset_free(scde_b200_ctx *ctx, scde_b200_dataset *ds);

/* scde.expression.magnitude: out[g + G*c] = (log(counts[g + G*c]) - corr_b[c]) / corr_a[c] */
SCDE_B200_API int scde_b200_expression_magnitude(scde_b200_ctx *ctx, const int32_t *counts, int32_t n_genes, int32_t n_cells,
                                   const double *corr_b, const double *corr_a, double *out);

/* ---- input preparation next to the path ---------------------------------------------------- */
/* scde.failure.probability (R/functions.R:725-750) for a genes x cells matrix: drop-out probability of every (gene, cell)
 * at the cell's magnitude -- taken from `magnitudes` (n_genes x n_cells, natural log) or, when that is NULL, from `counts`
 * as scde.expression.magnitude gives it.  models: n_cells x 12 (conc.a2 used when square_logit_conc).  NaN -> 0. */
SCDE_B200_API int scde_b200_failure_probability(scde_b200_ctx *ctx, const double *models, int32_t n_cells, const int32_t *counts,
                                  const double *magnitudes, int32_t n_genes, int32_t square_logit_conc, double *out);
/* scde.expression.prior (R/functions.R:225-254): magnitudes and drop-out weights of every (gene, cell), the max.quantile
 * quantile (type 7) of the finite magnitudes when max_value is NaN ("NULL"), stats::density (gaussian kernel, bandwidth
 * bw, weights, n = 2 length_out + 1, from -max_value to max_value) of the mirrored points, pseudo-count, normalisation.
 * Outputs, length_out + 1 values each: x (log10 scale), y, lp = log(y), grid_weight.  The O(genes x cells) work runs on
 * the device; the 2048-point kernel smoothing is host work. */
SCDE_B200_API int scde_b200_expression_prior(scde_b200_ctx *ctx, const double *models, int32_t n_cells, const int32_t *counts,
                               int32_t n_genes, int32_t square_logit_conc, int32_t length_out, double pseudo_count, double bw,
                               double max_quantile, double max_value, double *x, double *y, double *lp, double *grid_weight);

/* ---- diagnostics --------------------------------------------------------------------------- */
/* One cell's log-posterior table (the reference's ucposteriors[[i]]): out[n_grid * n_counts], grid index
 * fastest; modes[n_counts] (may be NULL).  n_cells_for_clamp sets the lower clamp -DBL_MAX/n/1.1. */
SCDE_B200_API int scde_b200_cell_table(scde_b200_ctx *ctx, const double *model_row12, const int32_t *unique_counts,
                         int32_t n_counts, const double *magnitudes, int32_t n_grid, int32_t local_theta,
                         int32_t square_logit_conc, int32_t n_cells_for_clamp, double *out, int32_t *modes);
/* The table of n_cells cells as the differential-expression call builds it for the tcgen05 contraction (zero-base form,
 * fixed-point planes, the context's options): models[n_cells x 12] column-major; each cell's distinct counts ascending in
 * ucl_flat[ucl_offsets[c] .. ucl_offsets[c + 1]), with or without a 0.  Outputs:
 *   q_out[n_rows][512 * ceil(n_grid / 102)]  the planes of every row, in the layout of scde_b200_probe_contract_i8: a
 *                                            zero-count row holds lp(0), every other row lp(x) - lp(0) of its cell (lp(x)
 *                                            when the cell is not based), up to a constant per row; "log 0" digits are 0;
 *   row_range_out[n_rows]                    first | last << 16 grid point that is not "log 0", or 0xFFFFFFFF;
 *   zero_row_out[n_cells], based_out[n_cells] the cell's zero-count row (-1: none) and whether that row is free of "log 0";
 *   zero_rows_out[n_cells][n_grid]           the zero-count row in FP64 (NaN for a cell without one).
 * n_rows = ucl_offsets[n_cells] >= 1; n_grid <= 408 (SCDE_B200_EINVAL otherwise: no fixed-point table exists). */
SCDE_B200_API int scde_b200_probe_table(scde_b200_ctx *ctx, const double *models, int32_t n_cells, const int32_t *ucl_flat,
                         const int32_t *ucl_offsets, const double *magnitudes, int32_t n_grid, int32_t local_theta,
                         int32_t square_logit_conc, int32_t n_cells_for_clamp, int8_t *q_out, uint32_t *row_range_out,
                         int32_t *zero_row_out, int32_t *based_out, double *zero_rows_out);
/* Measured FP64 FMA throughput of this device (TFLOP/s) from a register-resident DFMA loop; the roofline
 * denominator for the contraction kernel (MEASURED_PEAKS.json has no FP64 entry). */
SCDE_B200_API int scde_b200_measure_fp64_peak(scde_b200_ctx *ctx, double *tflops);
/* Contraction kernel of the bootstrap joint posterior: 0 = pick automatically (the tcgen05 fixed-point kernel where it
 * applies: K <= 408 grid points, zero-base table, multiplicities <= 127, every (gene, boot) keeps at least one grid point
 * that no drawn row marks "log 0" -- otherwise FP64); 1 = generic FP64 kernel; 2 = tiled FP64 kernel (mma.sync DMMA, exact
 * to rounding); 3 = tcgen05.mma kind::i8 fixed-point kernel (the table is rounded to 2^-29, sums are exact integers; error
 * if it does not apply at all, FP64 rerun if the data leave its range). */
SCDE_B200_API int scde_b200_set_contract_kernel(scde_b200_ctx *ctx, int32_t which);
/* Probe of the tcgen05 contraction kernel alone, on caller-made operands (tests): qtable[n_rows][512 * ceil(n_grid / 102)]
 * int8 in the layout [piece of 102 grid points][plane 0..4][102] (+ 2 zero bytes per piece); row_range[n_rows] (may be
 * NULL) = first | last << 16 grid point of the row that is not "log 0"; w8[n_w_rows][128] int8; entry lists as
 * (row, W row) with ld_lst a multiple of 32 and entries beyond lst_len[g] up to the next multiple of 32 pointing at an
 * all-zero W row.
 * t_out[n_genes][104][416] = 2^-29 * sum_p 256^p (sum_e plane_p[row_e][k] * w8[cell_e][b]), or -1e300 where a drawn row
 * is "log 0"; *flags_out (may be NULL) = the kernel's status word (4: a (gene, boot) without any admissible grid point). */
SCDE_B200_API int scde_b200_probe_contract_i8(scde_b200_ctx *ctx, const int8_t *qtable, int32_t n_rows, int32_t n_grid,
                                const uint32_t *row_range, const int8_t *w8, int32_t n_w_rows, const int32_t *lst_row,
                                const int32_t *lst_cell, const int32_t *lst_len, int32_t n_genes, int32_t ld_lst,
                                double *t_out, int32_t *flags_out);
/* scde_b200_probe_table plus qbound_out[n_rows][128]: the bound row of every fixed-point row (DESIGN.md 4.3, "Pruned
 * pieces"; layout in csrc/common.cuh), as the differential-expression call writes it. */
SCDE_B200_API int scde_b200_probe_table_bounds(scde_b200_ctx *ctx, const double *models, int32_t n_cells, const int32_t *ucl_flat,
                         const int32_t *ucl_offsets, const double *magnitudes, int32_t n_grid, int32_t local_theta,
                         int32_t square_logit_conc, int32_t n_cells_for_clamp, int8_t *q_out, uint32_t *row_range_out,
                         int32_t *zero_row_out, int32_t *based_out, double *zero_rows_out, int8_t *qbound_out);
/* scde_b200_probe_contract_i8 (t_out is the UNPRUNED T, without z) plus, when qbound (the bound rows of qtable) is given,
 * the pruning decision for the same launch: z[104][416] (or NULL: 0) is the zero-count base the soft-max would add;
 * lb_out[n_genes][104] the lower bound on every boot's row maximum, ub_out[n_genes][104][4] the upper bound on every
 * piece's admissible T (-inf: none), live_out[n_genes] bit p = piece p is contracted.  exp_out (may be NULL): exp_nonpos at
 * -745, -746 and -747 as the soft-max evaluates it on the device. */
SCDE_B200_API int scde_b200_probe_prune_i8(scde_b200_ctx *ctx, const int8_t *qtable, int32_t n_rows, int32_t n_grid,
                             const uint32_t *row_range, const int8_t *qbound, const double *z, const int8_t *w8,
                             int32_t n_w_rows, const int32_t *lst_row, const int32_t *lst_cell, const int32_t *lst_len,
                             int32_t n_genes, int32_t ld_lst, double *t_out, double *lb_out, double *ub_out,
                             uint8_t *live_out, double *exp_out, int32_t *flags_out);

#ifdef __cplusplus
}
#endif
#endif /* SCDE_B200_H */
