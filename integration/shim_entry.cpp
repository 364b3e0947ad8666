// shim_entry.cpp -- test wrapper (not part of what goes into the R package): builds the .Call arguments of
// scde_b200_diff and scde_b200_diff_contrasts (integration/scde_b200_shim.cpp) from plain arrays, calls it as R would, copies the result out.
// Linked into integration/_build/libscde_shim.so only (tests/test_gpu_parity.py).
#include <Rcpp.h>

#include <cstring>

RcppExport SEXP scde_b200_diff(SEXP Counts, SEXP Models, SEXP BatchModels, SEXP PriorX, SEXP PriorY, SEXP Group, SEXP Batch,
                               SEXP NBatchLevels, SEXP Nboot, SEXP Seed, SEXP ZeroIndex, SEXP ZeroIndexAdjusted,
                               SEXP LocalThetaFit, SEXP SquareLogitConc, SEXP Devices, SEXP DrawChunks);
RcppExport SEXP scde_b200_diff_contrasts(SEXP Counts, SEXP Models, SEXP BatchModels, SEXP PriorX, SEXP PriorY,
                                         SEXP GroupOffsets, SEXP GroupCells, SEXP Pairs, SEXP Batch, SEXP NBatchLevels,
                                         SEXP Nboot, SEXP Seed, SEXP ZeroIndex, SEXP ZeroIndexAdjusted, SEXP LocalThetaFit,
                                         SEXP SquareLogitConc, SEXP BatchLocalThetaFit, SEXP BatchSquareLogitConc,
                                         SEXP Devices, SEXP DrawChunks);

namespace {
SEXP ivec(const int *p, size_t n) {
    SEXP s = ShimArena::get().make(SHIM_INTSXP);
    s->ival.assign(p, p + n);
    return s;
}
SEXP dvec(const double *p, size_t n) {
    SEXP s = ShimArena::get().make(SHIM_REALSXP);
    s->dval.assign(p, p + n);
    return s;
}
}  // namespace

// no batch: out_idx[G*3] (as doubles, 0-based), out_z[G], out_cz[G]; with a batch factor additionally the batch.effect and
// batch.adjusted triples behind them (out arrays sized 3x).  draw_chunks: the DrawChunks argument (the reference's
// n.cores).  Returns 0, or -1 with the message in err[256].
extern "C" int shim_diff_chunked(const int *counts, int G, int C, const double *models12, const double *px, const double *py,
                                 int K, const int *group, const int *batch, int n_levels, int nboot, int zero_index,
                                 int zero_index_adj, const int *devices, int n_devices, int draw_chunks, double *out_idx,
                                 double *out_z, double *out_cz, char *err) {
    int rc = 0;
    try {
        SEXP cnt = ivec(counts, (size_t)G * C);
        cnt->nrow = G;
        cnt->ncol = C;
        SEXP mm = dvec(models12, (size_t)C * 12);
        mm->nrow = C;
        mm->ncol = 12;
        SEXP bm = dvec(models12, 0);
        bm->nrow = bm->ncol = 0;
        int one = 1, zero = 0;
        SEXP r = scde_b200_diff(cnt, mm, bm, dvec(px, K), dvec(py, K), ivec(group, C), ivec(batch, batch ? C : 0),
                                ivec(&n_levels, 1), ivec(&nboot, 1), ivec(&one, 1), ivec(&zero_index, 1),
                                ivec(&zero_index_adj, 1), ivec(&zero, 1), ivec(&zero, 1), ivec(devices, n_devices),
                                ivec(&draw_chunks, 1));
        const int n_sets = (int)r->list.size() / 3;
        for (int s = 0; s < n_sets; ++s) {
            std::memcpy(out_idx + (size_t)s * 3 * G, r->list[3 * s]->dval.data(), sizeof(double) * 3 * G);
            std::memcpy(out_z + (size_t)s * G, r->list[3 * s + 1]->dval.data(), sizeof(double) * G);
            std::memcpy(out_cz + (size_t)s * G, r->list[3 * s + 2]->dval.data(), sizeof(double) * G);
        }
    } catch (const std::exception &e) {
        std::strncpy(err, e.what(), 255);
        err[255] = 0;
        rc = -1;
    }
    ShimArena::get().clear();
    return rc;
}

// one draw set (n.cores = 1)
extern "C" int shim_diff(const int *counts, int G, int C, const double *models12, const double *px, const double *py, int K,
                         const int *group, const int *batch, int n_levels, int nboot, int zero_index, int zero_index_adj,
                         const int *devices, int n_devices, double *out_idx, double *out_z, double *out_cz, char *err) {
    return shim_diff_chunked(counts, G, C, models12, px, py, K, group, batch, n_levels, nboot, zero_index, zero_index_adj,
                             devices, n_devices, 1, out_idx, out_z, out_cz, err);
}

// scde_b200_diff_contrasts: groups as flattened 0-based cell lists, pairs[2 * n_contrasts]; batch models = models.
// out_idx[n_sets * n_contrasts * 3 * G] (as doubles), out_z / out_cz[n_sets * n_contrasts * G], n_sets = 3 with a batch
// factor (results, batch.effect, batch.adjusted), else 1; contrast c's block inside a set as in scde_b200_contrast_out.
extern "C" int shim_diff_contrasts_chunked(const int *counts, int G, int C, const double *models12, const double *px,
                                           const double *py, int K, const int *group_offsets, int n_groups,
                                           const int *group_cells, const int *pairs, int n_contrasts, const int *batch,
                                           int n_levels, int nboot, int zero_index, int zero_index_adj, const int *devices,
                                           int n_devices, int draw_chunks, double *out_idx, double *out_z, double *out_cz,
                                           char *err) {
    int rc = 0;
    try {
        SEXP cnt = ivec(counts, (size_t)G * C);
        cnt->nrow = G;
        cnt->ncol = C;
        SEXP mm = dvec(models12, (size_t)C * 12);
        mm->nrow = C;
        mm->ncol = 12;
        SEXP bm = dvec(models12, 0);
        bm->nrow = bm->ncol = 0;
        int one = 1, zero = 0;
        SEXP r = scde_b200_diff_contrasts(cnt, mm, bm, dvec(px, K), dvec(py, K), ivec(group_offsets, n_groups + 1),
                                          ivec(group_cells, group_offsets[n_groups]), ivec(pairs, 2 * (size_t)n_contrasts),
                                          ivec(batch, batch ? C : 0), ivec(&n_levels, 1), ivec(&nboot, 1), ivec(&one, 1),
                                          ivec(&zero_index, 1), ivec(&zero_index_adj, 1), ivec(&zero, 1), ivec(&zero, 1),
                                          ivec(&zero, 1), ivec(&zero, 1), ivec(devices, n_devices), ivec(&draw_chunks, 1));
        const int n_sets = (int)r->list.size() / 3;
        const size_t n3 = (size_t)3 * G * n_contrasts, n1 = (size_t)G * n_contrasts;
        for (int s = 0; s < n_sets; ++s) {
            std::memcpy(out_idx + s * n3, r->list[3 * s]->dval.data(), sizeof(double) * n3);
            std::memcpy(out_z + s * n1, r->list[3 * s + 1]->dval.data(), sizeof(double) * n1);
            std::memcpy(out_cz + s * n1, r->list[3 * s + 2]->dval.data(), sizeof(double) * n1);
        }
    } catch (const std::exception &e) {
        std::strncpy(err, e.what(), 255);
        err[255] = 0;
        rc = -1;
    }
    ShimArena::get().clear();
    return rc;
}

extern "C" int shim_diff_contrasts(const int *counts, int G, int C, const double *models12, const double *px, const double *py,
                                   int K, const int *group_offsets, int n_groups, const int *group_cells, const int *pairs,
                                   int n_contrasts, const int *batch, int n_levels, int nboot, int zero_index,
                                   int zero_index_adj, const int *devices, int n_devices, double *out_idx, double *out_z,
                                   double *out_cz, char *err) {
    return shim_diff_contrasts_chunked(counts, G, C, models12, px, py, K, group_offsets, n_groups, group_cells, pairs,
                                       n_contrasts, batch, n_levels, nboot, zero_index, zero_index_adj, devices, n_devices, 1,
                                       out_idx, out_z, out_cz, err);
}
