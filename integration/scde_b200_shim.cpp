// scde_b200_shim.cpp -- what a maintainer of the scde R package adds to src/ IN PLACE OF jpmatLogBoot.cpp and
// matSlideMult.cpp: the same five RcppExport symbols, with the same SEXP signatures, so that R/functions.R stays
// untouched -- .Call("logBootPosterior", ...) (R/functions.R:613,637), .Call("logBootBatchPosterior", ...) (:611,635),
// .Call("matSlideMult", ...) (:3545), .Call("jpmatLogBoot", ...) (:3535), .Call("jpmatLogBatchBoot", ...) (:3541) resolve
// to these functions, which call libscde_b200.so through its C ABI (include/scde_b200.h) -- plus .Call("scde_b200_diff",
// ...), the fused whole-path entry used by integration/scde_b200.R.
//
// Build inside the package: src/Makevars
//     PKG_CPPFLAGS += -I$(SCDE_B200_HOME)/include
//     PKG_LIBS     += -L$(SCDE_B200_HOME)/scde_b200 -lscde_b200 -Wl,-rpath,$(SCDE_B200_HOME)/scde_b200
// R is not installed in the authoring image; this file is nevertheless compiled and exercised there: the repository's
// header shim (oracle/shim/Rcpp.h) provides the subset of the Rcpp API used below, `make -C integration` links this
// file with the SEXP-building test wrappers of oracle/shim/ref_entry.cpp into integration/_build/libscde_shim.so, and
// tests/test_gpu_parity.py::test_r_shim_symbols_against_reference_fixtures drives the five symbols on a GPU and compares
// them with the reference's own C++ -- the code path an R session would take, minus R.
//
// Devices: SCDE_B200_DEVICES (e.g. "0,1,2,3") or the `devices` argument of scde_b200_diff selects the GPUs of a
// multi-device context, which shards the genes without changing results.  The reference's n.cores (the gene chunks of
// papply, R/functions.R:606-617, each with its own Seed) is the DrawChunks argument of the fused entries.
#include <Rcpp.h>
#include "scde_b200.h"

#include <cstdlib>
#include <string>
#include <vector>

namespace {

scde_b200_ctx *context(const std::vector<int> &devices = std::vector<int>()) {  // one context per R process
    static scde_b200_ctx *ctx = nullptr;
    static std::vector<int> have;
    std::vector<int> want = devices;
    if (want.empty()) {
        if (ctx) return ctx;
        if (const char *e = std::getenv("SCDE_B200_DEVICES")) {  // the shim's own switch (the library reads no environment)
            std::string s(e);
            size_t pos = 0;
            while (pos < s.size()) {
                size_t c = s.find(',', pos);
                if (c == std::string::npos) c = s.size();
                want.push_back(std::atoi(s.substr(pos, c - pos).c_str()));
                pos = c + 1;
            }
        }
        if (want.empty()) want.push_back(0);
    }
    if (ctx && want == have) return ctx;
    if (ctx) scde_b200_destroy(ctx);
    ctx = nullptr;
    if (scde_b200_create_multi((int)want.size(), want.data(), &ctx) != SCDE_B200_OK) Rcpp::stop(scde_b200_last_error());
    have = want;
    return ctx;
}

void check(int rc) {
    if (rc != SCDE_B200_OK) Rcpp::stop(scde_b200_last_error());
}

// list of integer vectors -> flat values + offsets (ucl, batchil)
void flatten(SEXP l, std::vector<int> &flat, std::vector<int> &off) {
    off.assign(1, 0);
    const int n = LENGTH(l);
    for (int i = 0; i < n; ++i) {
        Rcpp::IntegerVector v(VECTOR_ELT(l, i));
        flat.insert(flat.end(), v.begin(), v.end());
        off.push_back((int)flat.size());
    }
}

// jp (+ modes, + post as a list of C matrices G x K) as the reference returns them (src/jpmatLogBoot.cpp:277-330)
SEXP pack(int flag_modes, int flag_post, Rcpp::NumericMatrix jp, Rcpp::NumericMatrix modes, const std::vector<double> &post,
          int G, int C, int K) {
    if (!flag_modes && !flag_post) return jp;
    Rcpp::List pl(flag_post ? C : 0);
    for (int i = 0; i < (flag_post ? C : 0); ++i) {
        Rcpp::NumericMatrix m(G, K);
        std::copy(post.begin() + (size_t)i * G * K, post.begin() + (size_t)(i + 1) * G * K, m.begin());
        pl[i] = m;
    }
    if (flag_modes && flag_post)
        return Rcpp::List::create(Rcpp::Named("jp") = Rcpp::wrap(jp), Rcpp::Named("modes") = Rcpp::wrap(modes),
                                  Rcpp::Named("post") = Rcpp::wrap(pl));
    if (flag_modes) return Rcpp::List::create(Rcpp::Named("jp") = Rcpp::wrap(jp), Rcpp::Named("modes") = Rcpp::wrap(modes));
    return Rcpp::List::create(Rcpp::Named("jp") = Rcpp::wrap(jp), Rcpp::Named("post") = Rcpp::wrap(pl));
}

}  // namespace

// replaces src/jpmatLogBoot.cpp:100
RcppExport SEXP logBootPosterior(SEXP Models, SEXP Ucl, SEXP CountsI, SEXP Magnitudes, SEXP Nboot, SEXP Seed,
                                 SEXP ReturnIndividualPosteriors, SEXP LocalThetaFit, SEXP SquareLogitConc,
                                 SEXP EnsembleProbability) {
    Rcpp::NumericMatrix models(Models);  // C x 12, column-major, NA where a column is absent
    Rcpp::IntegerMatrix uci(CountsI);    // G x C, 0-based
    Rcpp::NumericVector mag(Magnitudes);
    std::vector<int> flat, off;
    flatten(Ucl, flat, off);
    const int G = uci.nrow(), C = uci.ncol(), K = mag.size(), flag = Rcpp::as<int>(ReturnIndividualPosteriors);
    const int fm = flag == 1 || flag == 3, fp = flag == 2 || flag == 3;
    Rcpp::NumericMatrix jp(G, K), modes(fm ? G : 0, fm ? C : 0);
    std::vector<double> post(fp ? (size_t)C * G * K : 0);
    check(scde_b200_log_boot_posterior(context(), models.begin(), C, flat.data(), off.data(), uci.begin(), G, mag.begin(), K,
                                       Rcpp::as<int>(Nboot), Rcpp::as<int>(Seed), /*boot_idx=*/NULL, flag,
                                       Rcpp::as<int>(LocalThetaFit), Rcpp::as<int>(SquareLogitConc),
                                       Rcpp::as<int>(EnsembleProbability), jp.begin(), fm ? modes.begin() : NULL,
                                       fp ? post.data() : NULL));
    return pack(fm, fp, jp, modes, post, G, C, K);
}

// replaces src/jpmatLogBoot.cpp:343
RcppExport SEXP logBootBatchPosterior(SEXP Models, SEXP Ucl, SEXP CountsI, SEXP Magnitudes, SEXP BatchIL, SEXP Composition,
                                      SEXP Nboot, SEXP Seed, SEXP ReturnIndividualPosteriors, SEXP LocalThetaFit,
                                      SEXP SquareLogitConc) {
    Rcpp::NumericMatrix models(Models);
    Rcpp::IntegerMatrix uci(CountsI);
    Rcpp::NumericVector mag(Magnitudes);
    Rcpp::IntegerVector comp(Composition);
    std::vector<int> flat, off, bflat, boff;
    flatten(Ucl, flat, off);
    flatten(BatchIL, bflat, boff);  // 0-based cell ids of every batch level (R/functions.R:570)
    const int G = uci.nrow(), C = uci.ncol(), K = mag.size(), flag = Rcpp::as<int>(ReturnIndividualPosteriors);
    const int fm = flag == 1, fp = flag == 2;  // the reference's batch function has no flag-3 branch (:501-530)
    Rcpp::NumericMatrix jp(G, K), modes(fm ? G : 0, fm ? C : 0);
    std::vector<double> post(fp ? (size_t)C * G * K : 0);
    if (bflat.empty()) bflat.push_back(0);
    check(scde_b200_log_boot_batch_posterior(context(), models.begin(), C, flat.data(), off.data(), uci.begin(), G, mag.begin(),
                                             K, comp.size(), boff.data(), bflat.data(), comp.begin(), Rcpp::as<int>(Nboot),
                                             Rcpp::as<int>(Seed), NULL, flag, Rcpp::as<int>(LocalThetaFit),
                                             Rcpp::as<int>(SquareLogitConc), jp.begin(), fm ? modes.begin() : NULL,
                                             fp ? post.data() : NULL));
    return pack(fm, fp, jp, modes, post, G, C, K);
}

// replaces src/matSlideMult.cpp:5
RcppExport SEXP matSlideMult(SEXP Mat1, SEXP Mat2) {
    Rcpp::NumericMatrix m1(Mat1), m2(Mat2);
    Rcpp::NumericMatrix out(m1.nrow(), 2 * m1.ncol() - 1);
    check(scde_b200_mat_slide_mult(context(), m1.begin(), m2.begin(), m1.nrow(), m1.ncol(), out.begin()));
    return out;
}

// replaces src/jpmatLogBoot.cpp:11 (legacy dense form; not divided by nboot, as the reference)
RcppExport SEXP jpmatLogBoot(SEXP Matl, SEXP Nboot, SEXP Seed) {
    const int nmat = LENGTH(Matl);
    Rcpp::NumericMatrix m0(VECTOR_ELT(Matl, 0));
    const int nrows = m0.nrow(), ncols = m0.ncol();
    std::vector<double> stack((size_t)nmat * nrows * ncols);
    for (int i = 0; i < nmat; ++i) {
        Rcpp::NumericMatrix m(VECTOR_ELT(Matl, i));
        std::copy(m.begin(), m.begin() + (size_t)nrows * ncols, stack.begin() + (size_t)i * nrows * ncols);
    }
    Rcpp::NumericMatrix jp(nrows, ncols);
    check(scde_b200_jpmat_log_boot(context(), stack.data(), nmat, nrows, ncols, Rcpp::as<int>(Nboot), Rcpp::as<int>(Seed), NULL,
                                   jp.begin()));
    return jp;
}

// replaces src/jpmatLogBoot.cpp:48
RcppExport SEXP jpmatLogBatchBoot(SEXP Matll, SEXP Comp, SEXP Nboot, SEXP Seed) {
    Rcpp::IntegerVector comp(Comp);
    const int nlev = LENGTH(Matll);
    Rcpp::NumericMatrix m0(VECTOR_ELT(VECTOR_ELT(Matll, 0), 0));
    const int nrows = m0.nrow(), ncols = m0.ncol();
    std::vector<int> off(1, 0);
    std::vector<double> stack;
    for (int k = 0; k < nlev; ++k) {
        SEXP pool = VECTOR_ELT(Matll, k);
        for (int i = 0; i < LENGTH(pool); ++i) {
            Rcpp::NumericMatrix m(VECTOR_ELT(pool, i));
            stack.insert(stack.end(), m.begin(), m.begin() + (size_t)nrows * ncols);
        }
        off.push_back(off.back() + LENGTH(pool));
    }
    Rcpp::NumericMatrix jp(nrows, ncols);
    check(scde_b200_jpmat_log_batch_boot(context(), stack.data(), nlev, off.data(), comp.begin(), nrows, ncols,
                                         Rcpp::as<int>(Nboot), Rcpp::as<int>(Seed), NULL, jp.begin()));
    return jp;
}

// The fused whole-path entry (scde_b200_expression_difference): counts in, grid indices and Z out; the joint posteriors
// never leave the device.  Called by scde.expression.difference.b200 (integration/scde_b200.R).
//   Counts   integer matrix genes x cells, columns in the order of the model rows
//   Models   numeric matrix cells x 12 (NA where a column is absent; corr.a already clamped to >= 1e-10)
//   Group    integer vector, 0 / 1 per cell, negative = NA;   Batch: integer codes 0..L-1 (negative = NA) or length 0
//   ZeroIndex / ZeroIndexAdjusted: 1-based H0 grid positions (length 1 or genes)
//   Devices  integer vector of CUDA device ids (length 0: SCDE_B200_DEVICES, else device 0); they do not change results
//   DrawChunks  the reference's n.cores: one draw set per gene chunk, Seed = Seed + the chunk's first gene (0-based)
//               (scde_b200_diff_args.draw_chunks; 1 = one draw set)
// Returns list(idx, z, cz[, batch.idx, batch.z, batch.cz, adjusted.idx, adjusted.z, adjusted.cz]).
RcppExport SEXP scde_b200_diff(SEXP Counts, SEXP Models, SEXP BatchModels, SEXP PriorX, SEXP PriorY, SEXP Group, SEXP Batch,
                               SEXP NBatchLevels, SEXP Nboot, SEXP Seed, SEXP ZeroIndex, SEXP ZeroIndexAdjusted,
                               SEXP LocalThetaFit, SEXP SquareLogitConc, SEXP Devices, SEXP DrawChunks) {
    Rcpp::IntegerMatrix counts(Counts);
    Rcpp::NumericMatrix models(Models), bmodels(BatchModels);
    Rcpp::NumericVector px(PriorX), py(PriorY);
    Rcpp::IntegerVector group(Group), batch(Batch), zi(ZeroIndex), zia(ZeroIndexAdjusted), devs(Devices);
    const int G = counts.nrow(), C = counts.ncol(), K = px.size();
    const bool has_batch = batch.size() == C && Rcpp::as<int>(NBatchLevels) > 1;
    scde_b200_diff_args a = scde_b200_diff_args();
    a.n_genes = G;
    a.n_cells = C;
    a.n_grid = K;
    a.counts = counts.begin();
    a.models = models.begin();
    a.prior_x = px.begin();
    a.prior_y = py.begin();
    a.group = group.begin();
    a.batch = has_batch ? batch.begin() : NULL;
    a.n_batch_levels = has_batch ? Rcpp::as<int>(NBatchLevels) : 0;
    a.n_boot = Rcpp::as<int>(Nboot);
    a.seed = Rcpp::as<int>(Seed);
    a.zero_index = zi.begin();
    a.n_zero = zi.size();
    a.zero_index_adjusted = zia.begin();
    a.local_theta = Rcpp::as<int>(LocalThetaFit);
    a.square_logit_conc = Rcpp::as<int>(SquareLogitConc);
    a.batch_models = (has_batch && bmodels.size() == C * 12) ? bmodels.begin() : NULL;
    a.batch_local_theta = a.local_theta;
    a.batch_square_logit_conc = a.square_logit_conc;
    a.draw_chunks = Rcpp::as<int>(DrawChunks);
    std::vector<int> idx((size_t)3 * G), bidx(has_batch ? (size_t)3 * G : 0), aidx(has_batch ? (size_t)3 * G : 0);
    Rcpp::NumericMatrix z(G, 1), bz(has_batch ? G : 0, 1), az(has_batch ? G : 0, 1);
    Rcpp::NumericMatrix cz(G, 1), bcz(has_batch ? G : 0, 1), acz(has_batch ? G : 0, 1);  // BH-corrected (R/functions.R:5051)
    scde_b200_diff_out o = scde_b200_diff_out();
    o.idx = idx.data();
    o.z = z.begin();
    o.cz = cz.begin();
    if (has_batch) {
        o.batch_idx = bidx.data();
        o.batch_z = bz.begin();
        o.batch_cz = bcz.begin();
        o.adjusted_idx = aidx.data();
        o.adjusted_z = az.begin();
        o.adjusted_cz = acz.begin();
    }
    std::vector<int> dv(devs.begin(), devs.end());
    check(scde_b200_expression_difference(context(dv), &a, &o, NULL));
    auto as_matrix = [G](const std::vector<int> &v) {  // G x 3 (lb, mle, ub), 0-based grid indices
        Rcpp::NumericMatrix m(G, 3);
        for (size_t i = 0; i < v.size(); ++i) m.begin()[i] = v[i];
        return m;
    };
    if (!has_batch)
        return Rcpp::List::create(Rcpp::Named("idx") = Rcpp::wrap(as_matrix(idx)), Rcpp::Named("z") = Rcpp::wrap(z),
                                  Rcpp::Named("cz") = Rcpp::wrap(cz));
    Rcpp::List out(9);  // idx, z, cz, batch.idx, batch.z, batch.cz, adjusted.idx, adjusted.z, adjusted.cz (named by the R wrapper)
    out[0] = as_matrix(idx);
    out[1] = z;
    out[2] = cz;
    out[3] = as_matrix(bidx);
    out[4] = bz;
    out[5] = bcz;
    out[6] = as_matrix(aidx);
    out[7] = az;
    out[8] = acz;
    return out;
}

// Many contrasts over one set of cells (scde_b200_dataset_*): the count matrix, its index and table are built once, each
// group's joint posterior once, and every contrast is what scde_b200_diff returns for the two groups (codes 0 / 1, every
// other cell NA).  Called by scde.expression.difference.contrasts.b200 (integration/scde_b200.R).
//   GroupOffsets / GroupCells  the groups as 0-based ascending cell lists, flattened (length n.groups + 1 / total)
//   Pairs                      2 x n.contrasts 0-based group ids, column c = (A, B) of contrast c
//   BatchModels                cells x 12 or a 0 x 0 matrix (= Models), with its own BatchLocalThetaFit / BatchSquareLogitConc
//                              flags (from colnames(batch.models))
//   DrawChunks                 as in scde_b200_diff, over the genes of Counts
// Returns list(idx, z, cz[, batch.idx, batch.z, batch.cz, adjusted.idx, adjusted.z, adjusted.cz]): idx genes x (3 x
// n.contrasts), contrast c in columns 3c+1 .. 3c+3 (lb, mle, ub, 0-based grid indices); z and cz genes x n.contrasts.
RcppExport SEXP scde_b200_diff_contrasts(SEXP Counts, SEXP Models, SEXP BatchModels, SEXP PriorX, SEXP PriorY,
                                         SEXP GroupOffsets, SEXP GroupCells, SEXP Pairs, SEXP Batch, SEXP NBatchLevels,
                                         SEXP Nboot, SEXP Seed, SEXP ZeroIndex, SEXP ZeroIndexAdjusted, SEXP LocalThetaFit,
                                         SEXP SquareLogitConc, SEXP BatchLocalThetaFit, SEXP BatchSquareLogitConc,
                                         SEXP Devices, SEXP DrawChunks) {
    Rcpp::IntegerMatrix counts(Counts);
    Rcpp::NumericMatrix models(Models), bmodels(BatchModels);
    Rcpp::NumericVector px(PriorX), py(PriorY);
    Rcpp::IntegerVector goff(GroupOffsets), gcells(GroupCells), pairs(Pairs), batch(Batch), zi(ZeroIndex),
        zia(ZeroIndexAdjusted), devs(Devices);
    const int G = counts.nrow(), C = counts.ncol(), K = px.size(), nc = pairs.size() / 2;
    const bool has_batch = batch.size() == C && Rcpp::as<int>(NBatchLevels) > 1;
    scde_b200_dataset_args d = scde_b200_dataset_args();
    d.n_genes = G;
    d.n_cells = C;
    d.n_grid = K;
    d.counts = counts.begin();
    d.models = models.begin();
    d.prior_x = px.begin();
    d.prior_y = py.begin();
    d.local_theta = Rcpp::as<int>(LocalThetaFit);
    d.square_logit_conc = Rcpp::as<int>(SquareLogitConc);
    scde_b200_contrast_args a = scde_b200_contrast_args();
    a.n_groups = goff.size() - 1;
    a.group_offsets = goff.begin();
    a.group_cells = gcells.begin();
    a.n_contrasts = nc;
    a.pairs = pairs.begin();
    a.n_boot = Rcpp::as<int>(Nboot);
    a.seed = Rcpp::as<int>(Seed);
    a.zero_index = zi.begin();
    a.n_zero = zi.size();
    a.zero_index_adjusted = zia.begin();
    a.batch = has_batch ? batch.begin() : NULL;
    a.n_batch_levels = has_batch ? Rcpp::as<int>(NBatchLevels) : 0;
    a.batch_models = (has_batch && bmodels.size() == C * 12) ? bmodels.begin() : NULL;
    a.batch_local_theta = Rcpp::as<int>(BatchLocalThetaFit);
    a.batch_square_logit_conc = Rcpp::as<int>(BatchSquareLogitConc);
    a.draw_chunks = Rcpp::as<int>(DrawChunks);
    const int n_sets = has_batch ? 3 : 1;
    std::vector<int> idx((size_t)n_sets * 3 * G * nc);
    std::vector<Rcpp::NumericMatrix> z, cz;
    for (int s = 0; s < n_sets; ++s) {
        z.push_back(Rcpp::NumericMatrix(G, nc));
        cz.push_back(Rcpp::NumericMatrix(G, nc));
    }
    scde_b200_contrast_out o = scde_b200_contrast_out();
    o.idx = idx.data();
    o.z = z[0].begin();
    o.cz = cz[0].begin();
    if (has_batch) {
        o.batch_idx = idx.data() + (size_t)3 * G * nc;
        o.batch_z = z[1].begin();
        o.batch_cz = cz[1].begin();
        o.adjusted_idx = idx.data() + (size_t)6 * G * nc;
        o.adjusted_z = z[2].begin();
        o.adjusted_cz = cz[2].begin();
    }
    std::vector<int> dv(devs.begin(), devs.end());
    scde_b200_ctx *ctx = context(dv);
    scde_b200_dataset *ds = NULL;
    check(scde_b200_dataset_create(ctx, &d, &ds, NULL));
    const int rc = scde_b200_dataset_contrasts(ctx, ds, &a, &o, NULL);
    const std::string msg = rc == SCDE_B200_OK ? std::string() : scde_b200_last_error();
    scde_b200_dataset_free(ctx, ds);  // before any R error: the context must accept the next call
    if (rc != SCDE_B200_OK) Rcpp::stop(msg);
    Rcpp::List out(3 * n_sets);  // named by the R wrapper
    for (int s = 0; s < n_sets; ++s) {
        Rcpp::NumericMatrix m(G, 3 * nc);
        for (size_t i = 0; i < (size_t)3 * G * nc; ++i) m.begin()[i] = idx[(size_t)s * 3 * G * nc + i];
        out[3 * s] = m;
        out[3 * s + 1] = z[s];
        out[3 * s + 2] = cz[s];
    }
    return out;
}
