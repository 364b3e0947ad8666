// lp_table.cu -- per-cell log-posterior rows (the reference's `ucposteriors`, src/jpmatLogBoot.cpp:128-211).
//
// For every (cell c, distinct count x) one table row of K grid values:
//   nb_k  = log NB(x; size = theta_k, prob = theta_k/(theta_k + mu~_k)) + log(1 - d_k)      (:166-188)
//   f     = log Pois(x; exp(fail.r))                                                         (:190)
//   v_k   = exp(nb_k - M) + exp(log d_k + f - M),  M = max(max_k nb_k, max_k log d_k + f)    (:191-193)
//   lp_k  = log(v_k / sum_j v_j), -Inf replaced by a finite sentinel                         (:194-204)
// with mu, d (drop-out probability) and theta from the cell's error-model row (:133-162) and the "snap" rule
// mu~_k = x when mu_k < x < mu_{k+1} (:173,182).  The negative-binomial / Poisson log-densities follow
// Loader's saddle-point algorithm as R's nmath evaluates them (stirlerr + bd0), so the table agrees with
// the reference's Rf_dnbinom / Rf_dpois to rounding error instead of suffering lgamma cancellation.
//
// Layout: one warp per row, lanes stride the grid; reductions over the grid are warp shuffles.  The
// k-independent pieces of the saddle-point formula (three stirlerr terms, two logs) are hoisted per row when
// theta is constant.  FP64 throughout.
#include "common.cuh"
#include "fastmath.cuh"
#include "ptx_sm100.cuh"
#include <cfloat>
#include <climits>
#include <cmath>
#include <cstdlib>

namespace scde {
namespace {

constexpr double LN_SQRT_2PI = 0.918938533204672741780329736406;
constexpr double LN_2PI = 1.837877066409345483560659472811;
constexpr double MIN_THETA = 1.0e-2, MAX_THETA = 1.0e+3;  // src/jpmatLogBoot.cpp:7-8

__constant__ double c_sferr_halves[31] = {
    0.0,
    0.1534264097200273452913848,   0.0810614667953272582196702,   0.0548141210519176538961390,
    0.0413406959554092940938221,   0.03316287351993628748511048,  0.02767792568499833914878929,
    0.02374616365629749597132920,  0.02079067210376509311152277,  0.01848845053267318523077934,
    0.01664469118982119216319487,  0.01513497322191737887351255,  0.01387612882307074799874573,
    0.01281046524292022692424986,  0.01189670994589177009505572,  0.01110455975820691732662991,
    0.010411265261972096497478567, 0.009799416126158803298389475, 0.009255462182712732917728637,
    0.008768700134139385462952823, 0.008330563433362871256469318, 0.007934114564314020547248100,
    0.007573675487951840794972024, 0.007244554301320383179543912, 0.006942840107209529865664152,
    0.006665247032707682442354394, 0.006408994188004207068439631, 0.006171712263039457647532867,
    0.005951370112758847735624416, 0.005746216513010115682023589, 0.005554733551962801371038690};

// log(n!) - log(sqrt(2 pi n) (n/e)^n)
__device__ double d_stirlerr(double n) {
    const double S0 = 0.083333333333333333333, S1 = 0.00277777777777777777778, S2 = 0.00079365079365079365079365,
                 S3 = 0.000595238095238095238095238, S4 = 0.0008417508417508417508417508;
    if (n <= 15.0) {
        double nn = n + n;
        if (nn == (double)(int)nn) return c_sferr_halves[(int)nn];
        return lgamma(n + 1.) - (n + 0.5) * log(n) + n - LN_SQRT_2PI;
    }
    double nn = n * n;
    if (n > 500) return (S0 - S1 / nn) / n;
    if (n > 80) return (S0 - (S1 - S2 / nn) / nn) / n;
    if (n > 35) return (S0 - (S1 - (S2 - S3 / nn) / nn) / nn) / n;
    return (S0 - (S1 - (S2 - (S3 - S4 / nn) / nn) / nn) / nn) / n;
}

// x log(x/np) + np - x without cancellation near x == np
__device__ double d_bd0(double x, double np) {
    if (!isfinite(x) || !isfinite(np) || np == 0.0) return nan("");
    if (fabs(x - np) < 0.1 * (x + np)) {
        double v = (x - np) / (x + np);
        double s = (x - np) * v;
        if (fabs(s) < DBL_MIN) return s;
        double ej = 2 * x * v;
        v = v * v;
        for (int j = 1; j < 1000; j++) {
            ej *= v;
            double s1 = s + ej / ((j << 1) + 1);
            if (s1 == s) return s1;
            s = s1;
        }
    }
    return x * log(x / np) + np - x;
}

__device__ double d_dbinom_raw_log(double x, double n, double p, double q) {
    if (p == 0) return (x == 0) ? 0.0 : -INFINITY;
    if (q == 0) return (x == n) ? 0.0 : -INFINITY;
    if (x == 0) {
        if (n == 0) return 0.0;
        return (p < 0.1) ? -d_bd0(n, n * q) - n * p : n * log(q);
    }
    if (x == n) return (q < 0.1) ? -d_bd0(n, n * p) - n * q : n * log(p);
    if (x < 0 || x > n) return -INFINITY;
    double lc = d_stirlerr(n) - d_stirlerr(x) - d_stirlerr(n - x) - d_bd0(x, n * p) - d_bd0(n - x, n * q);
    double lf = LN_2PI + log(x) + log1p(-x / n);
    return lc - 0.5 * lf;
}

// log dnbinom(x; size, prob), general form (used per grid point when theta varies along the grid)
__device__ double d_dnbinom_log(double x, double size, double prob) {
    if (isnan(x) || isnan(size) || isnan(prob)) return x + size + prob;
    if (prob <= 0 || prob > 1 || size < 0) return nan("");
    if (x < 0 || !isfinite(x)) return -INFINITY;
    if (x == 0 && size == 0) return 0.0;
    if (!isfinite(size)) size = DBL_MAX;
    if (x == 0) return size * log(prob);
    double ans = d_dbinom_raw_log(size, x + size, prob, 1 - prob);
    double p = size / (size + x);
    return log(p) + ans;
}

__device__ double d_dpois_log(double x, double lambda) {
    if (isnan(x) || isnan(lambda)) return x + lambda;
    if (lambda < 0) return nan("");
    if (x < 0 || !isfinite(x)) return -INFINITY;
    if (lambda == 0) return (x == 0) ? 0.0 : -INFINITY;
    if (!isfinite(lambda)) return -INFINITY;
    if (x <= lambda * DBL_MIN) return -lambda;
    if (lambda < x * DBL_MIN) return -lambda + x * log(lambda) - lgamma(x + 1);
    return -0.5 * log(2 * M_PI * x) + (-d_stirlerr(x) - d_bd0(x, lambda));
}

// Row-constant part of log dnbinom for fixed (x > 0, size): the same operations in the same order as
// d_dnbinom_log, with the k-independent terms evaluated once.
struct NbRow {
    double x, size, n, nmx, c1, half_lf, logp;
    bool regular;  // false -> fall back to the general function for every k
};
__device__ NbRow nb_row_prepare(double x, double size) {
    NbRow r;
    r.x = x;
    r.size = size;
    r.n = x + size;
    r.nmx = r.n - size;
    r.regular = (x > 0) && isfinite(x) && (size > 0) && isfinite(size) && !(size == r.n) && !(size > r.n);
    if (r.regular) {
        r.c1 = d_stirlerr(r.n) - d_stirlerr(size) - d_stirlerr(r.nmx);
        r.half_lf = 0.5 * (LN_2PI + log(size) + log1p(-size / r.n));
        r.logp = log(size / (size + x));
    } else {
        r.c1 = r.half_lf = r.logp = 0;
    }
    return r;
}
__device__ __forceinline__ double nb_row_eval(const NbRow &r, double prob) {
    if (!r.regular || !(prob > 0) || prob > 1) return d_dnbinom_log(r.x, r.size, prob);
    double q = 1 - prob;
    if (q == 0) return r.logp + -INFINITY;  // size != n here
    double lc = r.c1 - d_bd0(r.size, r.n * prob) - d_bd0(r.nmx, r.n * q);
    return r.logp + (lc - r.half_lf);
}

__device__ __forceinline__ double warp_max(double v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v = fmax(v, __shfl_xor_sync(0xffffffffu, v, o));
    return v;
}
__device__ __forceinline__ double warp_sum(double v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    return v;
}

// ---- per-cell grid vectors (src/jpmatLogBoot.cpp:133-162) ---------------------------------------
__global__ void cell_prep_kernel(const double *__restrict__ models, int ldm, int n_cells,
                                 const double *__restrict__ mag, int K, int local_theta, int sqlogit, CellPrep prep) {
    int c = blockIdx.x;
    if (c >= n_cells) return;
    int r = c;
    auto M = [&](int col) { return models[(size_t)col * ldm + r]; };
    const double corr_a = M(4), corr_b = M(3), conc_a = M(1), conc_b = M(0);
    const double conc_a2 = sqlogit ? M(11) : 0.0;
    double lmax = -INFINITY, csum = 0.0;
    for (int k = threadIdx.x; k < prep.ld; k += blockDim.x) {
        size_t o = (size_t)c * prep.ld + k;
        if (k >= K) {  // padding: benign values
            prep.mu[o] = 0;
            prep.lcfp[o] = 0;
            prep.lcfpr[o] = 0;
            if (prep.theta) prep.theta[o] = 1;
            if (prep.cfp) prep.cfp[o] = prep.l1[o] = prep.l2[o] = 0;
            continue;
        }
        double m = mag[k];
        double t = m * corr_a;
        t += corr_b;
        prep.mu[o] = exp(t);
        double cf;
        if (sqlogit) {
            cf = conc_a + m * conc_a2;
            cf *= m;
        } else {
            cf = m * conc_a;
        }
        cf += conc_b;
        cf = 1 / (exp(cf) + 1);
        double cr = 1 - cf;
        double l = log(cf);
        prep.lcfp[o] = l;
        prep.lcfpr[o] = log(cr);
        lmax = fmax(lmax, l);
        if (prep.cfp) {  // constant-theta fast path: log p_k, log q_k of the NB parametrisation and the drop-out prob
            const double th0 = M(5), muk = exp(t);
            prep.cfp[o] = cf;
            csum += cf;
            prep.l1[o] = -log1p(muk / th0);
            prep.l2[o] = -log1p(th0 / muk);
        }
        if (local_theta) {
            double th = -1 * m + M(8);
            th *= M(9);
            th = pow(10.0, th) + 1;
            th = pow(th, M(10));
            th = (M(7) - M(6)) / th;
            th += M(6);
            th = exp(-1 * th);
            if (!isfinite(th) || th < MIN_THETA) th = MIN_THETA;
            if (th > MAX_THETA) th = MAX_THETA;
            prep.theta[o] = th;
        }
    }
    __shared__ double red[32], red2[32];
    lmax = warp_max(lmax);
    csum = warp_sum(csum);
    if ((threadIdx.x & 31) == 0) {
        red[threadIdx.x >> 5] = lmax;
        red2[threadIdx.x >> 5] = csum;
    }
    __syncthreads();
    if (threadIdx.x < 32) {
        double v = threadIdx.x < (blockDim.x >> 5) ? red[threadIdx.x] : -INFINITY;
        double u = threadIdx.x < (blockDim.x >> 5) ? red2[threadIdx.x] : 0.0;
        v = warp_max(v);
        u = warp_sum(u);
        if (threadIdx.x == 0) {
            prep.maxcfp[c] = v;
            if (prep.scfp) prep.scfp[c] = u;
        }
    }
}

// ---- table rows ----------------------------------------------------------------------------------
constexpr int ROW_WARPS = 8;

__global__ void zero_rows_kernel(const int32_t *__restrict__ row_off, const int32_t *__restrict__ row_x, int n_cells,
                                 int32_t *__restrict__ zero_row, int64_t row_cap) {
    const int c = blockIdx.x;
    if (c >= n_cells) return;
    __shared__ int found;
    if (threadIdx.x == 0) found = -1;
    __syncthreads();
    // rows at or beyond the capacity do not exist (the chunked front's row estimate was too small: api.cu rebuilds)
    const int64_t end = min((int64_t)row_off[c + 1], row_cap);
    for (int64_t r = row_off[c] + threadIdx.x; r < end; r += blockDim.x)
        if (row_x[r] == 0) found = (int)r;  // a cell's distinct counts contain 0 at most once
    __syncthreads();
    if (threadIdx.x == 0) zero_row[c] = found;
}

__global__ void based_flags_kernel(const double *__restrict__ table, int ld_table, int K, double sentinel,
                                   const int32_t *__restrict__ zero_row, int n_cells, int32_t *__restrict__ based,
                                   int zero_compact_c0) {
    const int c = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
    if (c >= n_cells) return;
    const int lane = threadIdx.x & 31;
    const int zr = zero_row[c];
    bool ok = zr >= 0;
    // compact form (zero_compact_c0 >= 0): the FP64 table holds one row per CELL -- its zero-count row -- at the cell's index
    const size_t slot = zero_compact_c0 >= 0 ? (size_t)(zero_compact_c0 + c) : (size_t)(zr >= 0 ? zr : 0);
    if (ok)
        for (int k = lane; k < K; k += 32) {
            const double v = table[slot * ld_table + k];
            ok = ok && (v > sentinel) && isfinite(v);
        }
    ok = __all_sync(0xffffffffu, ok);
    if (lane == 0) based[c] = ok ? 1 : 0;
}

__global__ void row_cell_kernel(const int32_t *__restrict__ row_off, CellRange cr, int32_t *__restrict__ row_cell) {
    const int c = cr.c0 + blockIdx.x;
    if (c >= cr.c1) return;
    const int64_t end = min((int64_t)row_off[c + 1], cr.row_cap);
    for (int64_t r = row_off[c] + threadIdx.x; r < end; r += blockDim.x) row_cell[r] = c;
}

__global__ void __launch_bounds__(ROW_WARPS * 32)
lp_rows_kernel(const double *__restrict__ models, int ldm, CellRange cr, const int32_t *__restrict__ row_off,
               const int32_t *__restrict__ row_cell, const int32_t *__restrict__ row_x, CellPrep prep, int K, int local_theta,
               double sentinel,
               double *__restrict__ table, int ld_table, int32_t *__restrict__ row_mode, int which,
               const int32_t *__restrict__ zero_row, const int32_t *__restrict__ based) {
    extern __shared__ double s_buf[];  // ROW_WARPS x K
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    double *nb = s_buf + (size_t)warp * K;
    // items: the cells [c0, c1) (which == 1) or their table rows (bounds read here, on the device)
    const int64_t item0 = which == 1 ? (int64_t)cr.c0 : (int64_t)row_off[cr.c0];
    const int64_t item1 = which == 1 ? (int64_t)cr.c1 : min((int64_t)row_off[cr.c1], cr.row_cap);
    const int64_t n_items = item1 > item0 ? item1 - item0 : 0;
    // each CTA walks one contiguous run of rows, so consecutive rows of a warp belong to the same cell (or the next
    // one) and the per-cell grid vectors stay in L1
    const int64_t per_cta = (n_items + gridDim.x - 1) / gridDim.x;
    const int64_t item_end = item0 + min(n_items, (int64_t)(blockIdx.x + 1) * per_cta);
    for (int64_t item = item0 + (int64_t)blockIdx.x * per_cta + warp; item < item_end; item += ROW_WARPS) {
        int64_t row = item;
        int c;
        if (which == 1) {
            c = (int)item;
            row = zero_row[c];
            if (row < 0) continue;
        } else {
            c = row_cell[row];
            if (which == 2 && zero_row[c] == row) continue;
        }
        const double *zr = (which == 2 && based[c]) ? table + (size_t)zero_row[c] * ld_table : nullptr;
        const int mr = c;
        const double x = (double)row_x[row];
        const double *mu = prep.mu + (size_t)c * prep.ld;
        const double *lcfp = prep.lcfp + (size_t)c * prep.ld;
        const double *lcfpr = prep.lcfpr + (size_t)c * prep.ld;
        const double *thv = local_theta ? prep.theta + (size_t)c * prep.ld : nullptr;
        const double theta_c = models[(size_t)5 * ldm + mr];
        const double lambda = exp(models[(size_t)2 * ldm + mr]);
        NbRow nr;
        if (!local_theta) nr = nb_row_prepare(x, theta_c);
        double vmax = -INFINITY;
        for (int k = lane; k < K; k += 32) {
            double muv = mu[k];
            if ((k < K - 1 && x > muv && x < mu[k + 1]) || (k == K - 1 && x > muv)) muv = x;
            double v;
            if (local_theta) {
                double th = thv[k];
                v = d_dnbinom_log(x, th, th / (th + muv));
            } else if (x == 0) {
                double prob = theta_c / (theta_c + muv);
                v = (prob > 0 && prob <= 1 && theta_c >= 0 && isfinite(theta_c)) ? theta_c * log(prob)
                                                                                 : d_dnbinom_log(x, theta_c, prob);
            } else {
                v = nb_row_eval(nr, theta_c / (theta_c + muv));
            }
            v += lcfpr[k];
            nb[k] = v;
            vmax = fmax(vmax, v);
        }
        vmax = warp_max(vmax);
        const double fp = d_dpois_log(x, lambda);
        double maxp = vmax;
        const double alt = prep.maxcfp[c] + fp;
        if (maxp < alt) maxp = alt;
        double s = 0;
        for (int k = lane; k < K; k += 32) {
            double v = exp(nb[k] - maxp) + exp(lcfp[k] + fp - maxp);
            nb[k] = v;
            s += v;
        }
        s = warp_sum(s);
        double best = -INFINITY;
        int besti = 0x7fffffff;
        double *out = table + (size_t)row * ld_table;
        for (int k = lane; k < ld_table; k += 32) {
            if (k < K) {
                double v = log(nb[k] / s);
                if (besti == 0x7fffffff || v > best) {  // first maximum within this lane's ascending k
                    best = v;
                    besti = k;
                }
                if (v < sentinel) v = sentinel;
                out[k] = zr ? v - zr[k] : v;
            } else {
                out[k] = 0.0;
            }
        }
        // first maximum across lanes: larger value wins, ties go to the smaller index
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) {
            double ob = __shfl_xor_sync(0xffffffffu, best, o);
            int oi = __shfl_xor_sync(0xffffffffu, besti, o);
            if (ob > best || (ob == best && oi < besti) || (besti == 0x7fffffff && oi != 0x7fffffff)) {
                best = ob;
                besti = oi;
            }
        }
        if (lane == 0 && row_mode) row_mode[row] = (besti == 0x7fffffff) ? 0 : besti;
        __syncwarp();
    }
}

// ---- table rows, constant-theta fast path ---------------------------------------------------------
// With size = theta fixed along the grid the saddle-point form collapses: bd0(s, n p) + bd0(x, n q) =
// s log(s/n) + x log(x/n) - s log p - x log q (the linear terms cancel because p + q = 1), so
//     log NB(x; s, p_k) = R(x, s) + s * L1_k + x * L2_k,     L1_k = log p_k, L2_k = log q_k  (per cell, per grid point)
// with the row constant R = log(s/(s+x)) + stirlerr(n) - stirlerr(s) - stirlerr(n-s) - (log 2 pi + log s + log1p(-s/n))/2
//                           - s log(s/n) - x log1p(-s/n).
// Per element that is two FMAs, one exp (the drop-out term is cfp_k * exp(f - M)) and one log instead of two
// divisions, three logs and two exps.

// Row constants, one THREAD per row (the warp-per-row kernel below would execute this scalar code once per warp, i.e.
// 32 times more instruction issues): R(x, s), the "snap" pair log p / log q at mu~ = x, and the Poisson term.
__device__ __forceinline__ void row_const_one(const double *__restrict__ models, int ldm, const int32_t *__restrict__ row_cell,
                                              const int32_t *__restrict__ row_x, double4 *__restrict__ rowc,
                                              int32_t *__restrict__ row_snap, const double *__restrict__ mu_all,
                                              const double *__restrict__ lcfpr_all, int ld_mu, int K, int64_t row) {
    const int c = row_cell[row];
    const double x = (double)row_x[row];
    const double s = models[(size_t)5 * ldm + c];
    const double lambda = exp(models[(size_t)2 * ldm + c]);
    double R = 0.0, l1s = 0.0, l2s = 0.0;
    if (x > 0) {
        const double n = x + s, nmx = n - s;
        const double c1 = d_stirlerr(n) - d_stirlerr(s) - d_stirlerr(nmx);
        const double half_lf = 0.5 * (LN_2PI + log(s) + log1p(-s / n));
        R = log(s / (s + x)) + (c1 - half_lf) - (s * log(s / n) + nmx * log1p(-s / n));
        l1s = -log1p(x / s);  // "snap": mu~ = x
        l2s = -log1p(s / x);
    }
    // The snap rule (:173,182) replaces mu_k by x at the one grid point with mu_k < x < mu_{k+1} (or x > mu_{K-1} at the
    // last one).  mu_k = exp(corr.a m_k + corr.b) is non-decreasing along the grid (corr.a > 0), so that point is the last k
    // with mu_k < x: a binary search per row instead of two compares per table element.
    int ks = -1;
    if (x > 0) {
        const double *mu = mu_all + (size_t)c * ld_mu;
        int lo = -1, hi = K;
        while (hi - lo > 1) {
            const int mid = (lo + hi) >> 1;
            if (mu[mid] < x) lo = mid; else hi = mid;
        }
        if (lo == K - 1) ks = K - 1;
        else if (lo >= 0 && x < mu[lo + 1]) ks = lo;
    }
    row_snap[row] = ks;
    // (R, NB term at the snap point, the same + log(1 - d) at the snap grid point, Poisson term)
    const double snapv = fma(x, l2s, fma(s, l1s, R));
    rowc[row] = make_double4(R, snapv, ks >= 0 ? snapv + lcfpr_all[(size_t)c * ld_mu + ks] : -INFINITY, d_dpois_log(x, lambda));
}
__global__ void row_const_kernel(const double *__restrict__ models, int ldm, const int32_t *__restrict__ row_off,
                                 CellRange cr, const int32_t *__restrict__ row_cell, const int32_t *__restrict__ row_x,
                                 double4 *__restrict__ rowc, int32_t *__restrict__ row_snap, const double *__restrict__ mu_all,
                                 const double *__restrict__ lcfpr_all, int ld_mu, int K) {
    const int64_t row_end = min((int64_t)row_off[cr.c1], cr.row_cap);
    for (int64_t row = (int64_t)row_off[cr.c0] + (int64_t)blockIdx.x * blockDim.x + threadIdx.x; row < row_end;
         row += (int64_t)gridDim.x * blockDim.x)
        row_const_one(models, ldm, row_cell, row_x, rowc, row_snap, mu_all, lcfpr_all, ld_mu, K, row);
}

// Fixed-point planes (contract_i8.cu) of four consecutive table values: value = 2^-Q_FRAC * sum_p 256^p d_p with signed
// bytes d_p; values at or below the "log 0" sentinel get zero digits and a bit in `sent`.  x = rint(v 2^Q_FRAC) comes
// from the mantissa of v 2^Q_FRAC + 1.5 2^52; the balanced digits of x are the ordinary bytes of x + 0x8080808080 with the
// top bit of each flipped (adding 128 to every digit makes them ordinary base-256 digits); byte permutes transpose the four
// 32-bit words into one word per plane.  |v| <= 752 by construction (a difference of two values in [-752, 0]).
__device__ __forceinline__ void fixed_point_quad(const double (&v)[4], uint32_t (&word)[Q_NV], uint32_t &sent) {
    const double MAGIC = 6755399441055744.0;
    const long long BIAS = 0x8080808080ll;
    uint32_t lo[4], hi = 0u;
    sent = 0u;
#pragma unroll
    for (int e = 0; e < 4; ++e) {
        const double y = fma(v[e], (double)(1ll << Q_FRAC), MAGIC);
        long long x = __double_as_longlong(y) - __double_as_longlong(MAGIC) + BIAS;
        if (!(v[e] > -1.0e290)) {
            x = BIAS;
            sent |= 1u << e;
        }
        lo[e] = (uint32_t)x ^ 0x80808080u;
        hi |= (((uint32_t)(x >> 32) ^ 0x80u) & 0xFFu) << (8 * e);
    }
    const uint32_t t0 = __byte_perm(lo[0], lo[1], 0x5140), t1 = __byte_perm(lo[2], lo[3], 0x5140);
    const uint32_t t2 = __byte_perm(lo[0], lo[1], 0x7362), t3 = __byte_perm(lo[2], lo[3], 0x7362);
    word[0] = __byte_perm(t0, t1, 0x5410);
    word[1] = __byte_perm(t0, t1, 0x7632);
    word[2] = __byte_perm(t2, t3, 0x5410);
    word[3] = __byte_perm(t2, t3, 0x7632);
    word[4] = hi;
}
static_assert(Q_NV == 5, "fixed_point_quad is written for five value planes");
// byte offset of grid point k (even) in the row's fixed-point form [piece][plane][Q_PW]: plane 0 of its piece
__device__ __forceinline__ int q_offset(int k) {
    const int pc = (k >= Q_PW) + (k >= 2 * Q_PW) + (k >= 3 * Q_PW);
    return pc * Q_PIECE + (k - pc * Q_PW);
}

// The sweeps (one warp per row; lane l owns the grid points 4 l + 128 j .. + 3, so every access is a 16- or 32-byte
// vector and the index arithmetic is shared by four points; the row lives in a per-warp shared-memory buffer):
//   1. a_k = log NB_k + log(1 - d_k) and its maximum;  M = max(max_k a_k, max_k log d_k + f)          (:188-192)
//   2. S = sum_k exp(a_k - M) + exp(f - M) * sum_k d_k.  Terms with a_k - M <= -45 are below 3e-20 of S >= 1 and are
//      dropped; the drop-out part of the sum is one multiply (sum_k d_k comes from cell_prep).
//   3. lp_k = log(exp(a_k - M) + exp(log d_k + f - M)) - log S.  When one term exceeds the other by more than 37.5 nats
//      the smaller one is below half an ulp of the sum and log(exp(hi)) = hi, so no exp and no log is evaluated; in the
//      cross-over band, and below -708 where the reference's own exp() underflows gradually, the reference's expression
//      is evaluated as written (denormal rounding included); below -746 both exponentials are exactly 0 -> "log 0".
// Outputs: the FP64 table row (table, when write_f64) and / or its fixed-point planes and non-sentinel range (qtable,
// row_range); MODES: also row_mode.
// The reference's own expression for one table element, log(exp(nb - M) + exp(log d + f - M)) - log S with the clamp
// (:193-195,204): only evaluated in the cross-over and gradual-underflow bands.  Out of line, so that libm's exp / log
// (and their register demands) stay out of the row kernel's hot loop.
__device__ __noinline__ double lp_slow_element(double a, double dk, double lsum, double sentinel) {
    const double t = log(exp(a) + exp(dk)) - lsum;
    return t >= sentinel ? t : sentinel;
}

// LW lanes per row (32: one row per warp; 16: two rows per warp, side by side in the two half-warps -- 101 quads of a
// 401-point grid then occupy 7 x 16 = 112 lane slots instead of 4 x 32 = 128, every warp shuffle of the reductions serves
// two rows, and twice as many independent rows are in flight per warp).
// NORM = false: the row is stored without its normalising constant log S (sweep 2 is skipped).  A constant added to a
// whole table row adds a constant to T[b, :] of every (gene, boot) that draws the row, which the soft-max over the grid
// removes: the joint posterior cannot see it.  Only the fixed-point rows of the fused path are stored this way; FP64
// rows (zero-count rows, the `post` / cell-table outputs) are always normalised.
template <bool MODES, int LW, bool NORM>
__global__ void __launch_bounds__(ROW_WARPS * 32, LW == 32 ? 3 : 2)
lp_rows_fast_kernel(const double *__restrict__ models, int ldm, CellRange cr, const int32_t *__restrict__ row_off,
                    const int32_t *__restrict__ row_cell, const int32_t *__restrict__ row_x,
                    const double4 *__restrict__ rowc, const int32_t *__restrict__ row_snap, CellPrep prep, int K,
                    double sentinel, double *__restrict__ table, int ld_table, int32_t *__restrict__ row_mode, int which,
                    const int32_t *__restrict__ zero_row, const int32_t *__restrict__ based, int write_f64, int zero_compact,
                    int8_t *__restrict__ qtable, int ldq, uint32_t *__restrict__ row_range, int8_t *__restrict__ qbound) {
    constexpr int RPW = 32 / LW;  // rows per warp
    extern __shared__ __align__(16) unsigned char s_dyn[];
    double *s_rows = reinterpret_cast<double *>(s_dyn);                                  // [ROW_WARPS * RPW][KP_TILED]
    uint8_t *s_q = s_dyn + sizeof(double) * ROW_WARPS * RPW * KP_TILED;                  // [ROW_WARPS * RPW][4 * Q_PIECE]
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int h = lane / LW, l = lane % LW;
    double *nb = s_rows + (warp * RPW + h) * KP_TILED;
    uint8_t *sq = s_q + (warp * RPW + h) * (4 * Q_PIECE);
    if (qtable) {  // the two spare bytes of every piece, and the pieces beyond the grid, stay zero
        for (int j = l; j < (4 * Q_PIECE) / 4; j += LW) reinterpret_cast<uint32_t *>(sq)[j] = 0u;
        __syncwarp();
    }
    // items: the cells [c0, c1) (which == 1) or their table rows (bounds read here, on the device)
    const int64_t item0 = which == 1 ? (int64_t)cr.c0 : (int64_t)row_off[cr.c0];
    const int64_t item1 = which == 1 ? (int64_t)cr.c1 : min((int64_t)row_off[cr.c1], cr.row_cap);
    const int64_t n_items = item1 > item0 ? item1 - item0 : 0;
    const int kp = (K + 15) & ~15;
    // each CTA walks one contiguous run of rows, so consecutive rows of a warp belong to the same cell (or the next
    // one) and the per-cell grid vectors stay in L1
    const int64_t per_cta = (n_items + gridDim.x - 1) / gridDim.x;
    const int64_t item_end = item0 + min(n_items, (int64_t)(blockIdx.x + 1) * per_cta);
    // Row headers (row id, cell, count, row constants, snap point) are fetched one iteration ahead: they are dependent
    // global loads (row -> cell -> per-cell values) and were a quarter of the kernel's stall samples when fetched at the
    // top of the row's own iteration (profiles/r01w).
    struct Header {
        int64_t row;
        int c, ks;
        bool valid;
        double x;
        double4 rc;
    };
    auto load_header = [&](int64_t first) {
        // every lane runs the whole body (the reductions are full-warp shuffles); a half without a row of its own
        // recomputes a neighbour's and stores nothing
        Header hd;
        int64_t item = first + h;
        hd.valid = item < item_end;
        if (!hd.valid) item = item_end - 1;
        hd.row = item;
        if (which == 1) {
            hd.c = (int)item;
            hd.row = zero_row[hd.c];
            if (hd.row < 0) {  // no zero-count row (or it lies beyond the capacity): any existing row will do, nothing is stored
                hd.valid = false;
                hd.row = min((int64_t)row_off[hd.c], cr.row_cap - 1);
            }
        } else {
            hd.c = row_cell[hd.row];
        }
        hd.x = (double)row_x[hd.row];
        hd.rc = rowc[hd.row];
        hd.ks = row_snap[hd.row];
        return hd;
    };
    const int64_t first0 = item0 + (int64_t)blockIdx.x * per_cta + warp * RPW;
    Header nxt{};
    if (first0 < item_end) nxt = load_header(first0);
    for (int64_t first = first0; first < item_end; first += ROW_WARPS * RPW) {
        const Header cur = nxt;
        if (first + ROW_WARPS * RPW < item_end) nxt = load_header(first + ROW_WARPS * RPW);
        const int64_t row = cur.row;
        const int c = cur.c;
        bool valid = cur.valid;
        if (which == 2 && zero_row[c] == row) valid = false;
        const double *zr = (which == 2 && based[c]) ? table + (size_t)(zero_compact ? c : zero_row[c]) * ld_table : nullptr;
        const double x = cur.x;
        const double s = models[(size_t)5 * ldm + c];
        const size_t base = (size_t)c * prep.ld;
        const double *l1 = prep.l1 + base, *l2 = prep.l2 + base;
        const double *lcfpr = prep.lcfpr + base, *lcfp = prep.lcfp + base;
        const double R = cur.rc.x, snapv = cur.rc.y, fp = cur.rc.w;  // row constants from row_const_kernel
        const int ks = cur.ks;  // the grid point where mu~ snaps to x (:173,182), or -1
        // ---- sweep 1
        double vmax = -INFINITY;
        for (int k0 = 4 * l; k0 < K; k0 += 4 * LW) {
            double a1[4], a2[4], lr[4], v[4];
            *reinterpret_cast<double2 *>(&a1[0]) = *reinterpret_cast<const double2 *>(l1 + k0);
            *reinterpret_cast<double2 *>(&a1[2]) = *reinterpret_cast<const double2 *>(l1 + k0 + 2);
            *reinterpret_cast<double2 *>(&lr[0]) = *reinterpret_cast<const double2 *>(lcfpr + k0);
            *reinterpret_cast<double2 *>(&lr[2]) = *reinterpret_cast<const double2 *>(lcfpr + k0 + 2);
            if (x > 0) {
                *reinterpret_cast<double2 *>(&a2[0]) = *reinterpret_cast<const double2 *>(l2 + k0);
                *reinterpret_cast<double2 *>(&a2[2]) = *reinterpret_cast<const double2 *>(l2 + k0 + 2);
#pragma unroll
                for (int e = 0; e < 4; ++e) v[e] = fma(x, a2[e], fma(s, a1[e], R)) + lr[e];
#pragma unroll
                for (int e = 0; e < 4; ++e)
                    if (k0 + e == ks) v[e] = snapv + lr[e];
            } else {
#pragma unroll
                for (int e = 0; e < 4; ++e) v[e] = s * a1[e] + lr[e];
            }
#pragma unroll
            for (int e = 0; e < 4; ++e)
                if (k0 + e < K) vmax = fmax(vmax, v[e]);
#pragma unroll
            for (int e = 0; e < 4; ++e)
                if (k0 + e >= K) v[e] = -INFINITY;  // padding of the last quad (sweep 2 sums the whole quad)
            *reinterpret_cast<double2 *>(nb + k0) = make_double2(v[0], v[1]);
            *reinterpret_cast<double2 *>(nb + k0 + 2) = make_double2(v[2], v[3]);
        }
#pragma unroll
        for (int o = LW / 2; o > 0; o >>= 1) vmax = fmax(vmax, __shfl_xor_sync(0xffffffffu, vmax, o));
        double maxp = vmax;
        const double alt = prep.maxcfp[c] + fp;
        if (maxp < alt) maxp = alt;
        __syncwarp();
        // ---- sweep 2
        double lsum = 0.0;
        if (NORM) {
            double sum = 0;
            for (int k0 = 4 * l; k0 < K; k0 += 4 * LW) {
                double v[4];
                *reinterpret_cast<double2 *>(&v[0]) = *reinterpret_cast<const double2 *>(nb + k0);
                *reinterpret_cast<double2 *>(&v[2]) = *reinterpret_cast<const double2 *>(nb + k0 + 2);
#pragma unroll
                for (int e = 0; e < 4; ++e) {
                    // terms more than 50 nats below the maximum enter as exp(-50) = 2e-22 (401 of them are below an ulp
                    // of S >= 1); the padding of the row buffer beyond K holds -Inf and enters the same way
                    sum += exp_nonpos<false>(fmax(v[e] - maxp, -50.0));
                }
            }
#pragma unroll
            for (int o = LW / 2; o > 0; o >>= 1) sum += __shfl_xor_sync(0xffffffffu, sum, o);
            sum += exp(fp - maxp) * prep.scfp[c];
            lsum = log(sum);
        }
        // ---- sweep 3
        double best = -INFINITY;
        int besti = 0x7fffffff;
        double *out = table + (size_t)((zero_compact && which == 1) ? (int64_t)c : row) * ld_table;  // compact: a row per cell
        uint32_t okmask = 0u;  // bit 4 j + e: grid point 4 l + 4 LW j + e is not "log 0" (j-th quad of this lane)
        int jq = 0;
        for (int k0 = 4 * l; k0 < kp; k0 += 4 * LW, ++jq) {
            double v[4] = {0.0, 0.0, 0.0, 0.0};
            if (k0 < K) {
                double a[4], dk[4], z[4] = {0.0, 0.0, 0.0, 0.0}, L[4];
                *reinterpret_cast<double2 *>(&a[0]) = *reinterpret_cast<const double2 *>(nb + k0);
                *reinterpret_cast<double2 *>(&a[2]) = *reinterpret_cast<const double2 *>(nb + k0 + 2);
                *reinterpret_cast<double2 *>(&dk[0]) = *reinterpret_cast<const double2 *>(lcfp + k0);
                *reinterpret_cast<double2 *>(&dk[2]) = *reinterpret_cast<const double2 *>(lcfp + k0 + 2);
                if (zr) {
                    *reinterpret_cast<double2 *>(&z[0]) = *reinterpret_cast<const double2 *>(zr + k0);
                    *reinterpret_cast<double2 *>(&z[2]) = *reinterpret_cast<const double2 *>(zr + k0 + 2);
                }
                bool slow = false;
#pragma unroll
                for (int e = 0; e < 4; ++e) {
                    a[e] -= maxp;
                    dk[e] = (dk[e] + fp) - maxp;
                    const double d = a[e] - dk[e];
                    const double hi = d > 0.0 ? a[e] : dk[e];
                    const bool dead = hi < -746.0;  // both exponentials underflow to exactly 0: "log 0"
                    const bool easy = hi >= -708.0 && fabs(d) > 37.5;
                    L[e] = dead ? sentinel : hi - lsum;  // finite and far above the sentinel unless dead
                    slow = slow || !(dead || easy);
                }
                if (slow) {  // cross-over or gradual-underflow band somewhere in this quad: as the reference writes it
#pragma unroll
                    for (int e = 0; e < 4; ++e) {
                        const double d = a[e] - dk[e];
                        const double hi = d > 0.0 ? a[e] : dk[e];
                        if (!(hi < -746.0) && !(hi >= -708.0 && fabs(d) > 37.5)) L[e] = lp_slow_element(a[e], dk[e], lsum, sentinel);
                    }
                }
#pragma unroll
                for (int e = 0; e < 4; ++e) {
                    if (k0 + e < K) {
                        if (MODES) {  // argmax of the row before the clamp (:198-202): "log 0" counts as -Inf
                            const double t = L[e] > sentinel ? L[e] : -INFINITY;
                            if (besti == 0x7fffffff || t > best) {
                                best = t;
                                besti = k0 + e;
                            }
                        }
                        v[e] = L[e] - z[e];
                    }
                }
            }
            if (write_f64 && valid) {
                *reinterpret_cast<double2 *>(out + k0) = make_double2(v[0], v[1]);
                *reinterpret_cast<double2 *>(out + k0 + 2) = make_double2(v[2], v[3]);
            }
            if (qtable && k0 < Q_MAX_K) {
                uint32_t word[Q_NV], sent;
                fixed_point_quad(v, word, sent);
                const int nk = K - k0;  // real grid points in this quad
                okmask |= (~sent & (nk >= 4 ? 0xFu : nk > 0 ? (1u << nk) - 1u : 0u)) << (4 * jq);
                // pairs (k0, k0 + 1) and (k0 + 2, k0 + 3) never straddle a piece (Q_PW is even): 16-bit stores
                uint16_t *dst0 = reinterpret_cast<uint16_t *>(sq + q_offset(k0));
                uint16_t *dst1 = reinterpret_cast<uint16_t *>(sq + q_offset(k0 + 2));
#pragma unroll
                for (int p = 0; p < Q_NV; ++p) {
                    dst0[(p * Q_PW) >> 1] = (uint16_t)(word[p] & 0xFFFFu);
                    dst1[(p * Q_PW) >> 1] = (uint16_t)(word[p] >> 16);
                }
            }
        }
        if (write_f64 && valid)
            for (int k = kp + l; k < ld_table; k += LW) out[k] = 0.0;
        if (MODES) {
#pragma unroll
            for (int o = LW / 2; o > 0; o >>= 1) {
                double ob = __shfl_xor_sync(0xffffffffu, best, o);
                int oi = __shfl_xor_sync(0xffffffffu, besti, o);
                if (ob > best || (ob == best && oi < besti) || (besti == 0x7fffffff && oi != 0x7fffffff)) {
                    best = ob;
                    besti = oi;
                }
            }
        }
        __syncwarp();
        if (qtable) {  // the row's planes, 16 bytes per lane and store
            const uint4 *src = reinterpret_cast<const uint4 *>(sq);
            uint4 *dst = reinterpret_cast<uint4 *>(qtable + (size_t)row * ldq);
            if (valid)
                for (int j = l; j < ldq / 16; j += LW) dst[j] = src[j];
            // count, first and last of the grid points that are not "log 0" (bit b of a lane <-> k = 4 l + 4 LW (b >> 2) + (b & 3))
            int n_ok = __popc(okmask), kmin = 0x7fffffff, kmax = -1;
            if (okmask) {
                const int b0 = __ffs(okmask) - 1, b1 = 31 - __clz(okmask);
                kmin = 4 * l + 4 * LW * (b0 >> 2) + (b0 & 3);
                kmax = 4 * l + 4 * LW * (b1 >> 2) + (b1 & 3);
            }
#pragma unroll
            for (int o = LW / 2; o > 0; o >>= 1) {
                n_ok += __shfl_xor_sync(0xffffffffu, n_ok, o);
                kmin = min(kmin, __shfl_xor_sync(0xffffffffu, kmin, o));
                kmax = max(kmax, __shfl_xor_sync(0xffffffffu, kmax, o));
            }
            const uint32_t rr = (n_ok > 0 && kmax - kmin + 1 == n_ok) ? ((uint32_t)kmin | ((uint32_t)kmax << 16)) : Q_RANGE_IRREGULAR;
            if (l == 0 && valid) row_range[row] = rr;
            if (qbound && valid) q_bound_row(reinterpret_cast<const int8_t *>(sq), K, rr, qbound + (size_t)row * Q_BW, l, LW);
        }
        __syncwarp();
        if (MODES && l == 0 && valid) row_mode[row] = (besti == 0x7fffffff) ? 0 : besti;
    }
}

// ---- fixed-point rows of the fused path, cell state in registers -----------------------------------
// The rows the tcgen05 contraction reads (non-zero counts of a constant-theta model, stored in fixed point only, as the
// difference to the cell's zero-count row and without a normalising constant) are 99.9 % of the table.  For them a
// table element is   hi_k - Z_k,   hi_k = max(a_k, E_k + f) - M,   a_k = R + A_k + x L_k
// with the per-cell grid vectors A = theta log p + log(1 - d), L = log q, E = log d, Z = lp(0) and the row constants R, f,
// M -- everything a row adds is three scalars.  One warp walks a contiguous run of rows (consecutive rows belong to the
// same cell) and keeps A, L, E, Z of its 13 grid points per lane in registers, so the two sweeps of a row (maximum, then
// values) read nothing from memory: the kernel that loads the vectors per element (lp_rows_fast_kernel) spends 14 vector
// loads / stores per four elements and ~105 instructions per element, this one ~30.
//   Lane l owns the quads 4 (l + 32 j) .. + 3 for j < 3 (grid points 0..383) and the single point 384 + l: 13 points per
// lane, 416 per warp, so a 401-point grid uses 96 % of the lane slots (quads alone: 4 rounds for 101 quads = 79 %).
//   Row headers (count, row constants, snap point and its value) are loaded 32 rows at a time, one row per lane, one
// batch ahead, and broadcast by shuffles.
// Fixed point: y = v 2^29 + (1.5 2^52 + 0x8080808080) holds the biased digits of rint(v 2^29) in the low 40 bits of its
// mantissa (|v| <= 753, so 0 <= rint(v 2^29) + 0x8080808080 < 2^40); flipping the top bit of every byte gives the signed
// radix-256 digits.
using namespace ptx;
constexpr int QR_WARPS = 4;
constexpr int QR_MAIN = 3;  // quads per lane
constexpr int QR_CHUNK = 64;  // rows per work chunk (two header batches)

__device__ __forceinline__ double warp_max_redux(double v) {
    // order-preserving map double -> (hi, lo) unsigned, maximum by two 32-bit redux.sync
    const long long b = __double_as_longlong(v);
    uint32_t hi = (uint32_t)((unsigned long long)b >> 32), lo = (uint32_t)b;
    const uint32_t neg = (uint32_t)((int32_t)hi >> 31);  // all ones for negative values
    hi ^= neg | 0x80000000u;
    lo ^= neg;
    const uint32_t mh = __reduce_max_sync(0xffffffffu, hi);
    const uint32_t ml = __reduce_max_sync(0xffffffffu, hi == mh ? lo : 0u);
    const uint32_t back = (mh & 0x80000000u) ? 0x80000000u : 0xffffffffu;  // was non-negative : was negative
    const uint32_t rh = mh ^ back, rl = ml ^ ((mh & 0x80000000u) ? 0u : 0xffffffffu);
    return __longlong_as_double((long long)(((unsigned long long)rh << 32) | rl));
}

// row headers of one batch of 32 rows, staged by cp.async (two batches per warp)
struct QrHeaders {
    double4 rc[32];  // (R, -, value at the snap point, Poisson term)
    int32_t c[32], x[32], ks[32], pad[32];
};
// E = log d and Z = lp(0) of the lane's points are read once per element: they live in shared memory, [2 j + half][lane]
// as 16-byte pairs (every lane reads back what it wrote; consecutive lanes are consecutive: no bank conflicts), the
// single point in [2 QR_MAIN][lane].x
struct QrCell {
    double2 E[2 * QR_MAIN + 1][32], Z[2 * QR_MAIN + 1][32];
};
constexpr int QR_SMEM_WARP = 4 * Q_PIECE + 2 * (int)sizeof(QrHeaders) + (int)sizeof(QrCell) + Q_BW;  // + the staged bound row

// one slot of the staged bound row (common.cuh): its two digits
__device__ __forceinline__ void st_bound_slot(uint32_t sb, int slot, int v) {
    const int lo = (int)(int8_t)(v & 0xFF);
    st_shared_u8(sb + slot, (uint32_t)lo);
    st_shared_u8(sb + Q_BSLOTS + slot, (uint32_t)((v - lo) >> 8));
}
// x / 2^24 rounded up (CEIL) or down, x = rint(v 2^29) from the biased word of the digit trick below: with xb = x +
// 0x8080808080 = 2^24 A + r, x / 2^24 = A - 0x8080 + (r - 0x808080) / 2^24
template <bool CEIL>
__device__ __forceinline__ int q_bound_of(uint32_t lo, uint32_t hw) {
    const int t = (int)(__funnelshift_r(lo, hw, 24) & 0xFFFFu) - 0x8080;
    const uint32_t r = lo & 0xFFFFFFu;
    return CEIL ? t + (r > 0x808080u ? 1 : 0) : t - (r < 0x808080u ? 1 : 0);
}

// FULL: K >= 384, every quad of the three rounds lies inside the grid; BOUNDS: qbound != NULL (bound rows are written)
template <bool FULL, bool BOUNDS>
__global__ void __launch_bounds__(QR_WARPS * 32, 3)
lp_rows_q_kernel(const double *__restrict__ models, int ldm, CellRange cr, const int32_t *__restrict__ row_off,
                 const int32_t *__restrict__ row_cell, const int32_t *__restrict__ row_x,
                 const double4 *__restrict__ rowc, const int32_t *__restrict__ row_snap, CellPrep prep, int K,
                 double sentinel, const double *__restrict__ table, int ld_table, const int32_t *__restrict__ zero_row,
                 const int32_t *__restrict__ based, int8_t *__restrict__ qtable, int ldq, uint32_t *__restrict__ row_range,
                 unsigned long long *__restrict__ work_counter, int zero_compact, int8_t *__restrict__ qbound) {
    extern __shared__ __align__(16) unsigned char s_dyn[];  // [QR_WARPS][QR_SMEM_WARP]
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    uint8_t *sq = s_dyn + warp * QR_SMEM_WARP;
    QrHeaders *hdr = reinterpret_cast<QrHeaders *>(sq + 4 * Q_PIECE);
    QrCell *cell = reinterpret_cast<QrCell *>(sq + 4 * Q_PIECE + 2 * sizeof(QrHeaders));
    uint8_t *sbnd = sq + QR_SMEM_WARP - Q_BW;  // the row's bound row (common.cuh); its unused slots stay zero
    const uint32_t sb_addr = smem_u32(sbnd);
    for (int j = lane; j < (4 * Q_PIECE) / 16; j += 32) reinterpret_cast<uint4 *>(sq)[j] = make_uint4(0u, 0u, 0u, 0u);
    reinterpret_cast<uint32_t *>(sbnd)[lane] = 0u;
    __syncwarp();
    const int64_t row0 = (int64_t)row_off[cr.c0];
    const int64_t row1 = min((int64_t)row_off[cr.c1], cr.row_cap);
    const int64_t n_rows = row1 > row0 ? row1 - row0 : 0;
    // Rows are handed out in chunks of QR_CHUNK consecutive rows from a global counter (zeroed by the launcher): a warp
    // that starts late -- its CTA waited for room on an SM that another stream's kernel (the NCCL gather of the previous
    // step) was using -- or that meets slow rows simply takes fewer chunks.  With a static split of the rows over the
    // warps the slowest warp set the kernel's time (7.4 ms instead of 5.9 ms per rank at eight ranks).  Consecutive
    // chunks mostly belong to the same cell, whose grid vectors stay in registers across chunks.
    if (n_rows <= 0) return;
    const int64_t n_chunks = (n_rows + QR_CHUNK - 1) / QR_CHUNK;
    int64_t r_begin = 0, r_end = 0;

    // this lane's grid points and where their digits go in the staged row (shared-memory byte addresses)
    const int kt = 4 * 32 * QR_MAIN + lane;  // the single point
    const uint32_t sq_addr = smem_u32(sq);
    uint32_t off[QR_MAIN][2];
    uint32_t vmask = 0u;  // bit 4 j + e: main point (j, e) exists; bit 12: the single point exists
#pragma unroll
    for (int j = 0; j < QR_MAIN; ++j) {
        const int k0 = 4 * (lane + 32 * j);
        off[j][0] = sq_addr + q_offset(min(k0, Q_MAX_K - 2));
        off[j][1] = sq_addr + q_offset(min(k0 + 2, Q_MAX_K - 2));
#pragma unroll
        for (int e = 0; e < 4; ++e)
            if (k0 + e < K) vmask |= 1u << (4 * j + e);
    }
    if (kt < K) vmask |= 1u << (4 * QR_MAIN);
    uint32_t offt = sq_addr + q_offset(min(kt, Q_MAX_K - 1));
#pragma unroll
    for (int j = 0; j < QR_MAIN; ++j) asm volatile("" : "+r"(off[j][0]), "+r"(off[j][1]));  // keep them in registers
    asm volatile("" : "+r"(offt));

    // cell state
    double A[4 * QR_MAIN + 1], L[4 * QR_MAIN + 1];
    const bool tail_ok = kt < K;
    int cur_c = -1;
    int64_t cur_zero = -1;
    double maxcfp = 0.0;
    const double DEAD_FILL = -1.0e300;  // points beyond the grid: far below every threshold, never the maximum

    auto fetch_headers = [&](int64_t base, int slot) {  // one row per lane
        int64_t row = base + lane;
        if (row >= r_end) row = r_end - 1;
        QrHeaders *h = hdr + slot;
        cp_async16(smem_u32(&h->rc[lane]), &rowc[row]);
        cp_async16(smem_u32(&h->rc[lane]) + 16, reinterpret_cast<const char *>(&rowc[row]) + 16);
        cp_async4(smem_u32(&h->c[lane]), &row_cell[row]);
        cp_async4(smem_u32(&h->x[lane]), &row_x[row]);
        cp_async4(smem_u32(&h->ks[lane]), &row_snap[row]);
        cp_async_commit();
    };

    const double SCALE = (double)(1ll << Q_FRAC);
    const double MAGICB = 6755399441055744.0 + 551911719040.0;  // 1.5 2^52 + 0x8080808080
    constexpr uint32_t H_DEAD = 0xC0875000u, H_LOW = 0xC0862000u, H_BAND = 0x4042C000u;  // high words of -746, -708, 37.5
    for (;;) {
    unsigned long long ch = 0;
    if (lane == 0) ch = atomicAdd(work_counter, 1ull);
    ch = __shfl_sync(0xffffffffu, ch, 0);
    if ((int64_t)ch >= n_chunks) break;
    r_begin = row0 + (int64_t)ch * QR_CHUNK;
    r_end = min(row0 + n_rows, r_begin + QR_CHUNK);
    fetch_headers(r_begin, 0);
    int slot = 0;
    for (int64_t base = r_begin; base < r_end; base += 32, slot ^= 1) {
        if (base + 32 < r_end) {
            fetch_headers(base + 32, slot ^ 1);
            cp_async_wait<1>();
        } else {
            cp_async_wait<0>();
        }
        __syncwarp();
        const QrHeaders *h = hdr + slot;
        const int nb = (int)min((int64_t)32, r_end - base);
        for (int i = 0; i < nb; ++i) {
            const int64_t row = base + i;
            const int c = h->c[i];
            if (c != cur_c) {  // next cell: reload the grid vectors of this lane's points
                cur_c = c;
                const double theta = models[(size_t)5 * ldm + c];
                maxcfp = prep.maxcfp[c];
                const int zr = zero_row[c];
                cur_zero = zr;
                const bool bs = zr >= 0 && based[c] != 0;
                const size_t pb = (size_t)c * prep.ld;
                const double *zrow = table + (size_t)(zero_compact ? c : (zr >= 0 ? zr : 0)) * ld_table;
                double Ev[4 * QR_MAIN + 2], Zv[4 * QR_MAIN + 2];
                Ev[4 * QR_MAIN + 1] = Zv[4 * QR_MAIN + 1] = 0.0;
#pragma unroll
                for (int p = 0; p < 4 * QR_MAIN + 1; ++p) {
                    const int k = p < 4 * QR_MAIN ? 4 * (lane + 32 * (p >> 2)) + (p & 3) : kt;
                    if (k < K) {
                        A[p] = fma(theta, prep.l1[pb + k], prep.lcfpr[pb + k]);
                        L[p] = prep.l2[pb + k];
                        Ev[p] = prep.lcfp[pb + k];
                        Zv[p] = bs ? zrow[k] : 0.0;
                    } else {
                        A[p] = DEAD_FILL;
                        L[p] = 0.0;
                        Ev[p] = DEAD_FILL;
                        Zv[p] = 0.0;
                    }
                }
#pragma unroll
                for (int t = 0; t < 2 * QR_MAIN + 1; ++t) {
                    cell->E[t][lane] = make_double2(Ev[2 * t], Ev[2 * t + 1]);
                    cell->Z[t][lane] = make_double2(Zv[2 * t], Zv[2 * t + 1]);
                }
            }
            if (row == cur_zero) continue;  // the zero-count row is an FP64 row (lp_rows_fast_kernel, which == 1)
            const double x = (double)h->x[i];
            const int ks = h->ks[i];
            const double4 rc = h->rc[i];
            const double R = rc.x, asnap = rc.z, fp = rc.w;
            // ---- sweep 1: the row maximum.  The snapped value (mu~ = x maximises the NB term) replaces a_ks and is not
            // below it, so max(regular values, snapped value) is the maximum of the row as the reference builds it.
            double vmax = asnap;
#pragma unroll
            for (int p = 0; p < 4 * QR_MAIN + 1; ++p) {
                const double a = fma(x, L[p], R) + A[p];
                vmax = a > vmax ? a : vmax;
            }
            vmax = warp_max_redux(vmax);
            const double alt = maxcfp + fp;
            const double maxp = vmax > alt ? vmax : alt;
            const double Rm = R - maxp, fm = fp - maxp, asn = asnap - maxp;
            // ---- sweep 2: values, digits.  hi = max(a, e) (both relative to the row maximum, so hi <= 0 up to rounding).
            // The classes of lp_rows_fast_kernel's sweep 3 are decided on the high words of hi and of d = a - e, on the safe
            // side: "dead" (hi < -746: log 0) only when the high word alone proves it, "easy" (hi >= -708 and
            // |d| > 37.5: the value is hi) likewise; everything else -- the cross-over and gradual-underflow bands, and
            // the 1e-10-wide margins of the high-word tests -- evaluates the reference's expression as written.
            uint32_t okmask = 0u;
            const int qs = ks >> 2;  // (-1 -> -1: no quad)
            const int js = qs >> 5, es = ks & 3;
            const bool snap_lane = lane == (qs & 31);
#pragma unroll
            for (int j = 0; j < QR_MAIN; ++j) {
                double a[4], e[4], hi[4], z[4];
                {
                    const double2 e0 = cell->E[2 * j][lane], e1 = cell->E[2 * j + 1][lane];
                    const double2 z0 = cell->Z[2 * j][lane], z1 = cell->Z[2 * j + 1][lane];
                    e[0] = e0.x + fm, e[1] = e0.y + fm, e[2] = e1.x + fm, e[3] = e1.y + fm;
                    z[0] = z0.x, z[1] = z0.y, z[2] = z1.x, z[3] = z1.y;
                }
#pragma unroll
                for (int q = 0; q < 4; ++q) a[q] = fma(x, L[4 * j + q], Rm) + A[4 * j + q];
                if (js == j) {  // warp-uniform: the snap point lies in this round
#pragma unroll
                    for (int q = 0; q < 4; ++q) a[q] = (snap_lane && es == q) ? asn : a[q];
                }
                // alive bits per element; the slow band is looked for per quad first (all four "easy": nothing to do),
                // per element only inside the branch
                uint32_t alive = 0u, hh_max = 0u, band_min = 0xffffffffu;
                double d[4];
#pragma unroll
                for (int q = 0; q < 4; ++q) {
                    d[q] = a[q] - e[q];
                    const uint32_t hd = (uint32_t)__double2hiint(d[q]);
                    hi[q] = (int32_t)hd >= 0 ? a[q] : e[q];  // a >= e (for a - e == -0 the two are equal)
                    const uint32_t hh = (uint32_t)__double2hiint(hi[q]);
                    alive |= hh <= H_DEAD ? (1u << q) : 0u;
                    hh_max = max(hh_max, hh);
                    band_min = min(band_min, hd & 0x7fffffffu);
                }
                if (alive != 0u && !(hh_max < H_LOW && band_min > H_BAND)) {
                    if (hh_max < H_LOW) {
                        // cross-over band only, no exponential underflows: log(exp(a) + exp(e)) = hi + log1p(exp(-|d|)) to
                        // 1e-13 (for the quad's elements outside the band the correction is below their last bit)
#pragma unroll
                        for (int q = 0; q < 4; ++q)
                            hi[q] += log1p_unit(exp_nonpos<false>(fmax(-fabs(d[q]), -50.0)));
                    } else {
#pragma unroll
                        for (int q = 0; q < 4; ++q) {
                            const uint32_t hh = (uint32_t)__double2hiint(hi[q]);
                            const uint32_t hd = (uint32_t)__double2hiint(d[q]);
                            if (hh <= H_DEAD && !(hh < H_LOW && (hd & 0x7fffffffu) > H_BAND)) {
                                if ((hd & 0x7fffffffu) > H_BAND) {
                                    // gradual-underflow band, one term: the other exponential is exactly 0 (it lies 37.5
                                    // below a value under -708), so the reference's element is log(exp(hi)) with exp()
                                    // rounded to a denormal -- or log 0
                                    const double y = exp_nonpos<true>(hi[q]);
                                    hi[q] = log_tiny(y);
                                    if (!(y > 0.0)) alive &= ~(1u << q);
                                } else {
                                    hi[q] = lp_slow_element(a[q], e[q], 0.0, sentinel);
                                    if (!(hi[q] > sentinel)) alive &= ~(1u << q);
                                }
                            }
                        }
                    }
                }
                okmask |= alive << (4 * j);
                uint32_t lo[4], hw[4];
#pragma unroll
                for (int q = 0; q < 4; ++q) {
                    const long long yb = __double_as_longlong(fma(hi[q] - z[q], SCALE, MAGICB));
                    lo[q] = (uint32_t)yb;
                    hw[q] = (uint32_t)((unsigned long long)yb >> 32);
                }
                if (BOUNDS) {  // bound row: block 8 j + lane / 4 = the quads of lanes 4 (lane / 4) .. + 3; LB sample at 4 Q + 2
                    int ub = INT_MIN;
#pragma unroll
                    for (int q = 0; q < 4; ++q)
                        if ((alive >> q) & 1u) ub = max(ub, q_bound_of<true>(lo[q], hw[q]));
                    ub = max(ub, __shfl_xor_sync(0xffffffffu, ub, 1));
                    ub = max(ub, __shfl_xor_sync(0xffffffffu, ub, 2));
                    if ((lane & 3) == 0) st_bound_slot(sb_addr, 8 * j + (lane >> 2), ub == INT_MIN ? 0 : ub);
                    const int Q = lane + 32 * j;  // LB sample c at grid point 12 c + 6 = 4 (3 c + 1) + 2
                    if (Q % 3 == 1) st_bound_slot(sb_addr, Q_UB_N + (Q - 1) / 3, (alive >> 2) & 1u ? q_bound_of<false>(lo[2], hw[2]) : 0);
                }
                // byte q of every plane word belongs to element q: 0xFF where it is alive (dead elements store zero digits)
                const uint32_t am = ((alive * 0x00204081u) & 0x01010101u) * 0xFFu;
                const uint32_t t0 = __byte_perm(lo[0], lo[1], 0x5140), t1 = __byte_perm(lo[2], lo[3], 0x5140);
                const uint32_t t2 = __byte_perm(lo[0], lo[1], 0x7362), t3 = __byte_perm(lo[2], lo[3], 0x7362);
                uint32_t word[Q_NV];
                word[0] = (__byte_perm(t0, t1, 0x5410) ^ 0x80808080u) & am;
                word[1] = (__byte_perm(t0, t1, 0x7632) ^ 0x80808080u) & am;
                word[2] = (__byte_perm(t2, t3, 0x5410) ^ 0x80808080u) & am;
                word[3] = (__byte_perm(t2, t3, 0x7632) ^ 0x80808080u) & am;
                word[4] = (__byte_perm(__byte_perm(hw[0], hw[1], 0x0040), __byte_perm(hw[2], hw[3], 0x0040), 0x5410) ^ 0x80808080u) & am;
                const int k0 = 4 * (lane + 32 * j);
                if (FULL || k0 < K) {
#pragma unroll
                    for (int p = 0; p < Q_NV; ++p) st_shared_u16(off[j][0] + p * Q_PW, word[p]);
                }
                if (FULL || k0 + 2 < K) {
#pragma unroll
                    for (int p = 0; p < Q_NV; ++p) st_shared_u16(off[j][1] + p * Q_PW, word[p] >> 16);
                }
            }
            {  // the single point
                constexpr int P = 4 * QR_MAIN;
                double a = fma(x, L[P], Rm) + A[P];
                const double e = cell->E[2 * QR_MAIN][lane].x + fm;
                a = ks == kt ? asn : a;
                const uint32_t hd = (uint32_t)__double2hiint(a - e);
                double hi = (int32_t)hd >= 0 ? a : e;
                const uint32_t hh = (uint32_t)__double2hiint(hi);
                bool live = hh <= H_DEAD;
                if (live && !(hh < H_LOW && (hd & 0x7fffffffu) > H_BAND)) {
                    if ((hd & 0x7fffffffu) > H_BAND) {
                        const double y = exp_nonpos<true>(hi);
                        hi = log_tiny(y);
                        live = y > 0.0;
                    } else {
                        hi = lp_slow_element(a, e, 0.0, sentinel);
                        live = hi > sentinel;
                    }
                }
                const long long yb = __double_as_longlong(fma(hi - cell->Z[2 * QR_MAIN][lane].x, SCALE, MAGICB));
                const uint32_t am = live ? 0xFFFFFFFFu : 0u;
                const uint32_t lo = ((uint32_t)yb ^ 0x80808080u) & am, h8 = ((uint32_t)((unsigned long long)yb >> 32) ^ 0x80u) & am;
                okmask |= live ? (1u << P) : 0u;
                if (BOUNDS) {  // blocks 24 and 25: the single points of lanes 0..15 and 16..31
                    const uint32_t ylo = (uint32_t)yb, yhw = (uint32_t)((unsigned long long)yb >> 32);
                    int ub = live && tail_ok ? q_bound_of<true>(ylo, yhw) : INT_MIN;
#pragma unroll
                    for (int o = 1; o < 16; o <<= 1) ub = max(ub, __shfl_xor_sync(0xffffffffu, ub, o));
                    if ((lane & 15) == 0) st_bound_slot(sb_addr, 3 * 8 + (lane >> 4), ub == INT_MIN ? 0 : ub);
                    if (kt % Q_LB_STEP == Q_LB_OFF)
                        st_bound_slot(sb_addr, Q_UB_N + kt / Q_LB_STEP, live && tail_ok ? q_bound_of<false>(ylo, yhw) : 0);
                }
                if (tail_ok) {
                    st_shared_u8(offt, lo);
                    st_shared_u8(offt + Q_PW, lo >> 8);
                    st_shared_u8(offt + 2 * Q_PW, lo >> 16);
                    st_shared_u8(offt + 3 * Q_PW, lo >> 24);
                    st_shared_u8(offt + 4 * Q_PW, h8);
                }
            }
            okmask &= vmask;
            __syncwarp();
            {
                const uint4 *src = reinterpret_cast<const uint4 *>(sq) + lane;
                uint4 *dst = reinterpret_cast<uint4 *>(qtable + (size_t)row * ldq) + lane;
                if (FULL) {  // four pieces: 2048 bytes
                    const uint4 v0 = src[0], v1 = src[32], v2 = src[64], v3 = src[96];
                    dst[0] = v0, dst[32] = v1, dst[64] = v2, dst[96] = v3;
                } else {
                    for (int j = 0; j < ldq / 16 - lane; j += 32) dst[j] = src[j];
                }
                if (BOUNDS) reinterpret_cast<uint32_t *>(qbound + (size_t)row * Q_BW)[lane] = reinterpret_cast<const uint32_t *>(sbnd)[lane];
            }
            // count, first and last of the grid points that are not "log 0"; a lane's points ascend with the bit number:
            // bit b < 12 is grid point 4 lane + 128 (b >> 2) + (b & 3) = (4 lane - 96 (b >> 2)) + 32 b... written as
            // lane4 + 32 (b & 12) + (b & 3); bit 12 is 384 + lane
            const int lane4 = 4 * lane;
            const int b0 = __ffs(okmask) - 1, b1 = 31 - __clz(okmask);
            int kmin = b0 < 4 * QR_MAIN ? lane4 + 32 * (b0 & 12) + (b0 & 3) : kt;
            int kmax = b1 < 4 * QR_MAIN ? lane4 + 32 * (b1 & 12) + (b1 & 3) : kt;
            kmin = okmask ? kmin : 0x7fffffff;
            kmax = okmask ? kmax : -1;
            const int n_ok = __reduce_add_sync(0xffffffffu, __popc(okmask));
            kmin = __reduce_min_sync(0xffffffffu, kmin);
            kmax = __reduce_max_sync(0xffffffffu, kmax);
            if (lane == 0)
                row_range[row] = (n_ok > 0 && kmax - kmin + 1 == n_ok) ? ((uint32_t)kmin | ((uint32_t)kmax << 16))
                                                                        : Q_RANGE_IRREGULAR;
            __syncwarp();
        }
        __syncwarp();  // the headers of this slot are overwritten by the next iteration's fetch
    }
    }  // chunk loop
}

}  // namespace

cudaError_t launch_cell_prep(const double *models, int ld_models, int n_cells, const double *mag, int K,
                             int local_theta, int sqlogit, CellPrep prep, cudaStream_t st) {
    if (n_cells <= 0) return cudaSuccess;
    cell_prep_kernel<<<n_cells, 128, 0, st>>>(models, ld_models, n_cells, mag, K, local_theta, sqlogit, prep);
    return cudaGetLastError();
}

cudaError_t launch_row_cell(const int32_t *row_off, CellRange cr, int32_t *row_cell, cudaStream_t st) {
    if (cr.c1 <= cr.c0) return cudaSuccess;
    row_cell_kernel<<<cr.c1 - cr.c0, 128, 0, st>>>(row_off, cr, row_cell);
    return cudaGetLastError();
}

cudaError_t launch_row_consts(const double *models, int ld_models, const int32_t *row_off, CellRange cr,
                              const int32_t *row_cell, const int32_t *row_x, void *row_const, int32_t *row_snap,
                              CellPrep prep, int K, cudaStream_t st) {
    if (cr.c1 <= cr.c0) return cudaSuccess;
    const int blocks = min(148 * 16, 4 * (cr.c1 - cr.c0) + 1);  // grid-stride: the row count is only known on the device
    row_const_kernel<<<blocks, 256, 0, st>>>(models, ld_models, row_off, cr, row_cell, row_x, (double4 *)row_const, row_snap,
                                             prep.mu, prep.lcfpr, prep.ld, K);
    return cudaGetLastError();
}

cudaError_t launch_zero_rows(const int32_t *row_off, const int32_t *row_x, int n_cells, int32_t *zero_row, int64_t row_cap,
                             cudaStream_t st) {
    if (n_cells <= 0) return cudaSuccess;
    zero_rows_kernel<<<n_cells, 128, 0, st>>>(row_off, row_x, n_cells, zero_row, row_cap);
    return cudaGetLastError();
}

cudaError_t launch_based_flags(const double *table, int ld_table, int K, double sentinel, const int32_t *zero_row,
                               int n_cells, int32_t *based, cudaStream_t st, int zero_compact_c0) {
    if (n_cells <= 0) return cudaSuccess;
    based_flags_kernel<<<(n_cells + 7) / 8, 256, 0, st>>>(table, ld_table, K, sentinel, zero_row, n_cells, based,
                                                         zero_compact_c0);
    return cudaGetLastError();
}

cudaError_t launch_lp_rows(const double *models, int ld_models, CellRange cr, const int32_t *row_off,
                           const int32_t *row_cell_map, const int32_t *row_x, CellPrep prep, int K,
                           int local_theta, double sentinel, double *table, int ld_table, int32_t *row_mode, int which,
                           const int32_t *zero_row, const int32_t *based, void *row_const, const int32_t *row_snap,
                           int write_f64, int8_t *qtable, uint32_t *row_range, cudaStream_t st, int legacy_q_rows,
                           unsigned long long *work_counter, int zero_compact, int8_t *qbound) {
    if (cr.c1 <= cr.c0) return cudaSuccess;
    // compact FP64 table (one row per cell: its zero-count row): only the zero-count rows may be stored in FP64
    if (zero_compact && (which == 0 || (which == 2 && write_f64) || local_theta)) return cudaErrorInvalidValue;
    // the number of rows is only known on the device: size the grid for the cells (hundreds of rows each), grid-stride
    int64_t blocks = which == 1 ? ((int64_t)(cr.c1 - cr.c0) + ROW_WARPS - 1) / ROW_WARPS : (int64_t)(cr.c1 - cr.c0) * 8;
    const int64_t cap = 148 * 64;
    if (blocks > cap) blocks = cap;
    if (qtable && (!row_range || K > Q_MAX_K)) return cudaErrorInvalidValue;
    if (prep.cfp && prep.scfp && row_const && !local_theta && K <= KP_TILED && ld_table >= round_up(K, 16)) {
        if (!row_snap) return cudaErrorInvalidValue;
        if (which == 2 && qtable && !write_f64 && !row_mode && zero_row && based && prep.ld >= K && !legacy_q_rows) {
            // fixed-point rows only: the register-resident kernel; one contiguous run of rows per warp
            const size_t smem = (size_t)QR_WARPS * QR_SMEM_WARP;
            auto launch_q = [&](auto kernel) -> cudaError_t {
                cudaError_t e = cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
                if (e != cudaSuccess) return e;
                if (!work_counter) return cudaErrorInvalidValue;
                e = cudaMemsetAsync(work_counter, 0, sizeof(unsigned long long), st);
                if (e != cudaSuccess) return e;
                kernel<<<148 * 3, QR_WARPS * 32, smem, st>>>(models, ld_models, cr, row_off, row_cell_map, row_x,
                                                             (const double4 *)row_const, row_snap, prep, K, sentinel, table,
                                                             ld_table, zero_row, based, qtable, q_row_bytes(K), row_range,
                                                             work_counter, zero_compact, qtable ? qbound : nullptr);
                return cudaGetLastError();
            };
            if (qbound)
                return K >= 4 * 32 * QR_MAIN ? launch_q(lp_rows_q_kernel<true, true>) : launch_q(lp_rows_q_kernel<false, true>);
            return K >= 4 * 32 * QR_MAIN ? launch_q(lp_rows_q_kernel<true, false>) : launch_q(lp_rows_q_kernel<false, false>);
        }
        auto launch =[&](auto kernel, int rpw) -> cudaError_t {
            const size_t smem = (size_t)ROW_WARPS * rpw * (sizeof(double) * KP_TILED + 4 * Q_PIECE);
            cudaError_t e = cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
            if (e != cudaSuccess) return e;
            kernel<<<(unsigned)blocks, ROW_WARPS * 32, smem, st>>>(
                models, ld_models, cr, row_off, row_cell_map, row_x, (const double4 *)row_const, row_snap, prep, K, sentinel,
                table, ld_table, row_mode, which, zero_row, based, write_f64, zero_compact, qtable, q_row_bytes(K), row_range,
                qtable ? qbound : nullptr);
            return cudaGetLastError();
        };
        const bool norm = write_f64 != 0;  // rows that exist in fixed point only need no normalising constant
        if (row_mode)
            return norm ? launch(lp_rows_fast_kernel<true, 16, true>, 2) : launch(lp_rows_fast_kernel<true, 16, false>, 2);
        return norm ? launch(lp_rows_fast_kernel<false, 16, true>, 2) : launch(lp_rows_fast_kernel<false, 16, false>, 2);
    }
    if (qtable || !write_f64) return cudaErrorInvalidValue;  // the general kernel writes the FP64 table only
    size_t smem = (size_t)ROW_WARPS * K * sizeof(double);
    if (smem > 48 * 1024) {
        cudaError_t e = cudaFuncSetAttribute(lp_rows_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
        if (e != cudaSuccess) return e;
    }
    lp_rows_kernel<<<(unsigned)blocks, ROW_WARPS * 32, smem, st>>>(models, ld_models, cr, row_off, row_cell_map, row_x, prep, K,
                                                                  local_theta, sentinel, table, ld_table, row_mode, which,
                                                                  zero_row, based);
    return cudaGetLastError();
}

}  // namespace scde
