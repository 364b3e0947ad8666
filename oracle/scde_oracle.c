/*
 * scde_oracle.c -- CPU ORACLE for the scde differential-expression posterior path.
 *
 * TEST INFRASTRUCTURE ONLY.  Nothing in the product (scde_b200/, include/) may link,
 * import or call this file; only tests/, __graft_entry__.smoke() and bench.py's
 * cpu_baseline / --impl reference legs use it, and there only as the checker / CPU arm.
 *
 * PARITY STATUS: pinned against THE REFERENCE'S OWN C++ compiled here.  The reference ships no
 * assertions (tests/tests.R only checks that nothing throws, SURVEY.md section 4) and its build
 * needs R, Rcpp, RcppArmadillo (absent from the image) -- but its two translation units of this
 * path, src/jpmatLogBoot.cpp and src/matSlideMult.cpp, compile UNMODIFIED against the header shim
 * oracle/shim/RcppArmadillo.h (the part of R / Rcpp / Armadillo they use, restated; Makefile target
 * `ref` -> oracle/_ref/libscde_ref.so).  tests/test_ref.py holds every entry point of this file to
 * that library BIT FOR BIT (all returnpost forms, batch, ensemble, no-bootstrap, local theta, legacy
 * forms, matSlideMult, the rand() rejection loop; without the library, against the digests of its
 * outputs in tests/golden/ref_digests.json), and tests/golden/ref_fixtures_*.npz keeps outputs of
 * it.  What stays restated -- "parity unpinned" in the
 * strict sense -- is R itself: nmath's dnbinom / dpois (used by BOTH sides through Rf_dnbinom /
 * Rf_dpois of the shim), qnorm / pnorm / p.adjust and the R-level ratio-posterior / summary code
 * (R/functions.R), pinned by (a) mpmath 50-digit values, (b) scipy ndtri, (c) numpy.correlate,
 * (d) glibc srand/rand known answers, (e) the printed rows of vignettes/diffexp.md:113-119.
 *
 * This is a plain-C, FP64, single-threaded (per gene chunk) restatement, in the reference's
 * loop order, of
 *   src/jpmatLogBoot.cpp:100-331   logBootPosterior
 *   src/jpmatLogBoot.cpp:343-531   logBootBatchPosterior
 *   src/jpmatLogBoot.cpp:11-86     jpmatLogBoot / jpmatLogBatchBoot (legacy dense form)
 *   src/matSlideMult.cpp:5-23      matSlideMult
 *   R/functions.R:3491-3510        calculate.ratio.posterior
 *   R/functions.R:3514-3531        get.ratio.posterior.Z.score
 *   R/functions.R:5039-5053        quick.distribution.summary
 *   R/functions.R:694-697          scde.expression.magnitude
 * Third-party arithmetic the reference pulls from R (not in /root/reference; R >= 3.0.0,
 * DESCRIPTION:34, version unpinned) is restated from its published algorithms:
 *   dnbinom / dbinom_raw / dpois_raw / stirlerr / bd0  -- C. Loader (2000), "Fast and
 *       Accurate Computation of Binomial Probabilities", as used by R nmath;
 *   qnorm  -- Wichura (1988) AS 241 PPND16;   pnorm -- via erfc;
 *   rowSums / cumsum accumulate in long double (R's LDOUBLE on x86-64);
 *   p.adjust(method = "BH").
 * The bootstrap RNG is the platform libc srand()/rand() exactly as the reference calls it.
 *
 * Build: see oracle/Makefile (gcc -O2 -ffp-contract=off, R's default optimisation level,
 * no FMA contraction so results match an x86-64 R build without -march flags).
 */
#define _GNU_SOURCE /* qsort_r */
#include <float.h>
#include <math.h>
#include <stdint.h>
#include <stdlib.h>
#include <string.h>

#define MIN_THETA 1.0e-2 /* src/jpmatLogBoot.cpp:7 */
#define MAX_THETA 1.0e+3 /* src/jpmatLogBoot.cpp:8 */

/* model matrix columns, src/jpmatLogBoot.cpp:101-112 */
enum { CONCB_I = 0, CONCA_I, FAILR_I, CORRB_I, CORRA_I, CORRT_I,
       CORRLTB_I, CORRLTT_I, CORRLTM_I, CORRLTS_I, CORRLTR_I, CONCA2_I, NMODELCOL };

#define LN_SQRT_2PI 0.918938533204672741780329736406
#define LN_2PI 1.837877066409345483560659472811

/* ------------------------------------------------------------------------------------ */
/* Loader's saddle-point pieces (R nmath: stirlerr.c, bd0.c, dbinom.c, dpois.c, dnbinom.c) */

static const double sferr_halves[31] = {
    0.0,                           /* n=0 - wrong, place holder only */
    0.1534264097200273452913848,   /* 0.5 */
    0.0810614667953272582196702,   /* 1.0 */
    0.0548141210519176538961390,   /* 1.5 */
    0.0413406959554092940938221,   /* 2.0 */
    0.03316287351993628748511048,  /* 2.5 */
    0.02767792568499833914878929,  /* 3.0 */
    0.02374616365629749597132920,  /* 3.5 */
    0.02079067210376509311152277,  /* 4.0 */
    0.01848845053267318523077934,  /* 4.5 */
    0.01664469118982119216319487,  /* 5.0 */
    0.01513497322191737887351255,  /* 5.5 */
    0.01387612882307074799874573,  /* 6.0 */
    0.01281046524292022692424986,  /* 6.5 */
    0.01189670994589177009505572,  /* 7.0 */
    0.01110455975820691732662991,  /* 7.5 */
    0.010411265261972096497478567, /* 8.0 */
    0.009799416126158803298389475, /* 8.5 */
    0.009255462182712732917728637, /* 9.0 */
    0.008768700134139385462952823, /* 9.5 */
    0.008330563433362871256469318, /* 10.0 */
    0.007934114564314020547248100, /* 10.5 */
    0.007573675487951840794972024, /* 11.0 */
    0.007244554301320383179543912, /* 11.5 */
    0.006942840107209529865664152, /* 12.0 */
    0.006665247032707682442354394, /* 12.5 */
    0.006408994188004207068439631, /* 13.0 */
    0.006171712263039457647532867, /* 13.5 */
    0.005951370112758847735624416, /* 14.0 */
    0.005746216513010115682023589, /* 14.5 */
    0.005554733551962801371038690  /* 15.0 */
};

/* stirlerr(n) = log(n!) - log( sqrt(2*pi*n)*(n/e)^n ) */
double orc_stirlerr(double n) {
    const double S0 = 0.083333333333333333333;        /* 1/12 */
    const double S1 = 0.00277777777777777777778;      /* 1/360 */
    const double S2 = 0.00079365079365079365079365;   /* 1/1260 */
    const double S3 = 0.000595238095238095238095238;  /* 1/1680 */
    const double S4 = 0.0008417508417508417508417508; /* 1/1188 */
    double nn;
    if (n <= 15.0) {
        nn = n + n;
        if (nn == (int)nn) return sferr_halves[(int)nn];
        return lgamma(n + 1.) - (n + 0.5) * log(n) + n - LN_SQRT_2PI;
    }
    nn = n * n;
    if (n > 500) return (S0 - S1 / nn) / n;
    if (n > 80) return (S0 - (S1 - S2 / nn) / nn) / n;
    if (n > 35) return (S0 - (S1 - (S2 - S3 / nn) / nn) / nn) / n;
    return (S0 - (S1 - (S2 - (S3 - S4 / nn) / nn) / nn) / nn) / n;
}

/* bd0(x, np) = x log(x/np) + np - x, evaluated without cancellation near x == np */
double orc_bd0(double x, double np) {
    if (!isfinite(x) || !isfinite(np) || np == 0.0) return NAN;
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

/* log of the binomial point mass, real-valued x and n (dbinom_raw, give_log = TRUE) */
static double dbinom_raw_log(double x, double n, double p, double q) {
    double lf, lc;
    if (p == 0) return (x == 0) ? 0.0 : -INFINITY;
    if (q == 0) return (x == n) ? 0.0 : -INFINITY;
    if (x == 0) {
        if (n == 0) return 0.0;
        lc = (p < 0.1) ? -orc_bd0(n, n * q) - n * p : n * log(q);
        return lc;
    }
    if (x == n) {
        lc = (q < 0.1) ? -orc_bd0(n, n * p) - n * q : n * log(p);
        return lc;
    }
    if (x < 0 || x > n) return -INFINITY;
    lc = orc_stirlerr(n) - orc_stirlerr(x) - orc_stirlerr(n - x) - orc_bd0(x, n * p) - orc_bd0(n - x, n * q);
    lf = LN_2PI + log(x) + log1p(-x / n);
    return lc - 0.5 * lf;
}

/* Rf_dnbinom(x, size, prob, log = TRUE); call sites src/jpmatLogBoot.cpp:174,183,418,427 */
double orc_dnbinom_log(double x, double size, double prob) {
    if (isnan(x) || isnan(size) || isnan(prob)) return x + size + prob;
    if (prob <= 0 || prob > 1 || size < 0) return NAN;
    if (x < 0 || !isfinite(x)) return -INFINITY;
    if (x == 0 && size == 0) return 0.0;
    if (!isfinite(size)) size = DBL_MAX;
    if (x == 0) return size * log(prob); /* exact small-x limit; prob == 1 gives log 1 */
    double ans = dbinom_raw_log(size, x + size, prob, 1 - prob);
    double p = size / (size + x);
    return log(p) + ans;
}

/* Rf_dpois(x, lambda, log = TRUE); call sites src/jpmatLogBoot.cpp:190,432 */
double orc_dpois_log(double x, double lambda) {
    if (isnan(x) || isnan(lambda)) return x + lambda;
    if (lambda < 0) return NAN;
    if (x < 0 || !isfinite(x)) return -INFINITY;
    if (lambda == 0) return (x == 0) ? 0.0 : -INFINITY;
    if (!isfinite(lambda)) return -INFINITY;
    if (x <= lambda * DBL_MIN) return -lambda;
    if (lambda < x * DBL_MIN) return -lambda + x * log(lambda) - lgamma(x + 1);
    return -0.5 * log(2 * M_PI * x) + (-orc_stirlerr(x) - orc_bd0(x, lambda));
}

/* ------------------------------------------------------------------------------------ */
/* qnorm(p, lower.tail = FALSE) -- AS 241 PPND16; pnorm(x, lower.tail = FALSE) */

double orc_qnorm_upper(double p) {
    if (isnan(p)) return p;
    if (p < 0 || p > 1) return NAN;
    if (p == 0) return INFINITY;
    if (p == 1) return -INFINITY;
    double p_ = 0.5 - p + 0.5; /* lower-tail probability */
    double q = p_ - 0.5, r, val;
    if (fabs(q) <= 0.425) {
        r = .180625 - q * q;
        val = q * (((((((r * 2509.0809287301226727 + 33430.575583588128105) * r + 67265.770927008700853) * r +
                        45921.953931549871457) * r + 13731.693765509461125) * r + 1971.5909503065514427) * r +
                     133.14166789178437745) * r + 3.387132872796366608) /
              (((((((r * 5226.495278852854561 + 28729.085735721942674) * r + 39307.89580009271061) * r +
                   21213.794301586595867) * r + 5394.1960214247511077) * r + 687.1870074920579083) * r +
                42.313330701600911252) * r + 1.);
        return val;
    }
    r = (q < 0) ? p_ : p; /* min(p, 1-p), taken from the accurately known tail */
    r = sqrt(-log(r));
    if (r <= 5.) {
        r += -1.6;
        val = (((((((r * 7.7454501427834140764e-4 + .0227238449892691845833) * r + .24178072517745061177) * r +
                    1.27045825245236838258) * r + 3.64784832476320460504) * r + 5.7694972214606914055) * r +
                 4.6303378461565452959) * r + 1.42343711074968357734) /
              (((((((r * 1.05075007164441684324e-9 + 5.475938084995344946e-4) * r + .0151986665636164571966) * r +
                   .14810397642748007459) * r + .68976733498510000455) * r + 1.6763848301838038494) * r +
                2.05319162663775882187) * r + 1.);
    } else {
        r += -5.;
        val = (((((((r * 2.01033439929228813265e-7 + 2.71155556874348757815e-5) * r + .0012426609473880784386) * r +
                    .026532189526576123093) * r + .29656057182850489123) * r + 1.7848265399172913358) * r +
                 5.4637849111641143699) * r + 6.6579046435011037772) /
              (((((((r * 2.04426310338993978564e-15 + 1.4215117583164458887e-7) * r + 1.8463183175100546818e-5) * r +
                   7.868691311456132591e-4) * r + .0148753612908506148525) * r + .13692988092273580531) * r +
                .59983220655588793769) * r + 1.);
    }
    if (q < 0.0) val = -val;
    return val;
}

double orc_pnorm_upper(double x) { return 0.5 * erfc(x * M_SQRT1_2); }

/* ------------------------------------------------------------------------------------ */
/* bootstrap draws: libc srand/rand with the reference's rejection rule                 */

/* src/jpmatLogBoot.cpp:221,255-257: srand(seed); per boot, n draws rj = rand()/(RAND_MAX/n),
 * redrawn while rj >= n.  out[b*n + j] in draw order. */
void orc_boot_indices(int seed, int n, int nboot, int *out) {
    srand((unsigned)seed);
    for (int b = 0; b < nboot; b++)
        for (int j = 0; j < n; j++) {
            int rj;
            while (n <= (rj = rand() / (RAND_MAX / n)))
                ;
            out[(size_t)b * n + j] = rj;
        }
}

/* src/jpmatLogBoot.cpp:467,470-490: per boot, for each batch level k with comp[k] > 0, comp[k]
 * draws from pool k (same rule with n = pool size); the drawn value is mapped to the global
 * cell id bi[rj].  out[b*D + d], D = sum(comp), draw order preserved. */
void orc_batch_boot_indices(int seed, int nlevels, const int *pool_off, const int *pool_cells, const int *comp,
                            int nboot, int *out) {
    srand((unsigned)seed);
    size_t o = 0;
    for (int b = 0; b < nboot; b++)
        for (int k = 0; k < nlevels; k++) {
            int nsamp = comp[k];
            if (nsamp > 0) {
                const int *bi = pool_cells + pool_off[k];
                int ncells = pool_off[k + 1] - pool_off[k];
                for (int j = 0; j < nsamp; j++) {
                    int rj;
                    while (ncells <= (rj = rand() / (RAND_MAX / ncells)))
                        ;
                    out[o++] = bi[rj];
                }
            }
        }
}

/* ------------------------------------------------------------------------------------ */
/* per-cell log-posterior table, src/jpmatLogBoot.cpp:128-211 (batch: :373-457)          */

/* Armadillo's sum() of contiguous memory -- sum(vector) and every column of sum(M, 0) -- is arrayops::accumulate: two
 * interleaved partial sums, acc1 over the even and acc2 over the odd positions, returned as acc1 + acc2.  Restated
 * because the order decides the last bit; checked bit for bit against the reference compiled against the header shim
 * (oracle/_ref, tests/test_ref.py). */
static double arma_accumulate(const double *src, int n) {
    double acc1 = 0.0, acc2 = 0.0;
    int j;
    for (j = 1; j < n; j += 2) {
        acc1 += *src++;
        acc2 += *src++;
    }
    if ((j - 1) < n) acc1 += *src;
    return acc1 + acc2;
}

/* Fill pm[K x ncounts] (column j = grid vector for unique count uc[j], contiguous) and, if maxi != NULL,
 * the per-column argmax (first maximum, taken BEFORE the lower clamp as in :198-204). */
static void cell_table(const double *models, int ncells_total, int i, const int *uc, int ncounts, const double *mag,
                       int K, int localtheta, int squarelogitconc, double minlogprob, double *pm, int *maxi) {
#define M(col) models[(size_t)(col) * ncells_total + i]
    double *mu = (double *)malloc(sizeof(double) * K * 5);
    double *cfp = mu + K, *cfpr = cfp + K, *thetas = cfpr + K, *nbp = thetas + K;
    for (int k = 0; k < K; k++) { /* :133-134 */
        double t = mag[k] * M(CORRA_I);
        t += M(CORRB_I);
        mu[k] = exp(t);
    }
    double maxcfp = -INFINITY;
    for (int k = 0; k < K; k++) { /* :135-146 */
        double c;
        if (squarelogitconc) {
            c = M(CONCA_I) + mag[k] * M(CONCA2_I);
            c *= mag[k];
        } else {
            c = mag[k] * M(CONCA_I);
        }
        c += M(CONCB_I);
        c = 1 / (exp(c) + 1);
        double cr = 1 - c;
        cfp[k] = log(c);
        cfpr[k] = log(cr);
        if (k == 0 || cfp[k] > maxcfp) maxcfp = cfp[k]; /* :146 max(cfp) */
    }
    if (localtheta) { /* :148-162 */
        for (int k = 0; k < K; k++) {
            double t = -1 * mag[k] + M(CORRLTM_I);
            t *= M(CORRLTS_I);
            t = pow(10.0, t) + 1; /* arma::exp10 */
            t = pow(t, M(CORRLTR_I));
            t = (M(CORRLTT_I) - M(CORRLTB_I)) / t;
            t += M(CORRLTB_I);
            t = exp(-1 * t);
            if (!isfinite(t) || t < MIN_THETA) t = MIN_THETA;
            if (t > MAX_THETA) t = MAX_THETA;
            thetas[k] = t;
        }
    }
    double lambda = exp(M(FAILR_I));
    for (int j = 0; j < ncounts; j++) { /* :166-206 */
        double x = uc[j];
        for (int k = 0; k < K; k++) {
            double muv = mu[k];
            double theta = localtheta ? thetas[k] : M(CORRT_I);
            /* "snap" rule :173/:182 */
            if ((k < K - 1 && x > muv && x < mu[k + 1]) || (k == K - 1 && x > muv)) muv = x;
            nbp[k] = orc_dnbinom_log(x, theta, theta / (theta + muv));
        }
        for (int k = 0; k < K; k++) nbp[k] += cfpr[k]; /* :188 */
        double fp = orc_dpois_log(x, lambda);          /* :190 */
        double maxp = nbp[0];                          /* :191-192 */
        for (int k = 1; k < K; k++)
            if (nbp[k] > maxp) maxp = nbp[k];
        if (maxp < (maxcfp + fp)) maxp = maxcfp + fp;
        for (int k = 0; k < K; k++) /* :193 */
            nbp[k] = exp(nbp[k] - maxp) + exp(cfp[k] + fp - maxp);
        const double sd = arma_accumulate(nbp, K); /* :194 sum(nbp) */
        for (int k = 0; k < K; k++) nbp[k] = log(nbp[k] / sd); /* :194-195 */
        if (maxi) {                                             /* :198-202 first maximum */
            int mi = 0;
            double mv = nbp[0];
            for (int k = 1; k < K; k++)
                if (nbp[k] > mv) { mv = nbp[k]; mi = k; }
            maxi[j] = mi;
        }
        for (int k = 0; k < K; k++) /* :204 */
            if (nbp[k] < minlogprob) nbp[k] = minlogprob;
        memcpy(pm + (size_t)j * K, nbp, sizeof(double) * K); /* :205 */
    }
    free(mu);
#undef M
}

typedef struct {
    int ncells, K;
    double **pm; /* per cell: K x U_c */
    int **maxi;  /* per cell: U_c (or NULL) */
} table_t;

static void table_build(table_t *t, const double *models, int ncells, const int *ucl_flat, const int *ucl_off,
                        const double *mag, int K, int localtheta, int sqlogit, int want_modes) {
    t->ncells = ncells;
    t->K = K;
    t->pm = (double **)calloc(ncells, sizeof(double *));
    t->maxi = (int **)calloc(ncells, sizeof(int *));
    double minlogprob = -1 * DBL_MAX / ncells / 1.1; /* :127 (batch :372: ncells = all cells) */
    for (int i = 0; i < ncells; i++) {
        int nc = ucl_off[i + 1] - ucl_off[i];
        t->pm[i] = (double *)malloc(sizeof(double) * (size_t)K * (nc > 0 ? nc : 1));
        if (want_modes) t->maxi[i] = (int *)malloc(sizeof(int) * (nc > 0 ? nc : 1));
        cell_table(models, ncells, i, ucl_flat + ucl_off[i], nc, mag, K, localtheta, sqlogit, minlogprob, t->pm[i],
                   want_modes ? t->maxi[i] : NULL);
    }
}

static void table_free(table_t *t) {
    for (int i = 0; i < t->ncells; i++) {
        free(t->pm[i]);
        free(t->maxi[i]);
    }
    free(t->pm);
    free(t->maxi);
}

/* expose one cell's table for unit tests: out[K x ncounts] column-major (grid index fastest), modes[ncounts] */
void orc_cell_table(const double *model_row12, const int *uc, int ncounts, const double *mag, int K, int localtheta,
                    int sqlogit, int ncells_for_clamp, double *out, int *modes) {
    double minlogprob = -1 * DBL_MAX / ncells_for_clamp / 1.1;
    cell_table(model_row12, 1, 0, uc, ncounts, mag, K, localtheta, sqlogit, minlogprob, out, modes);
}

/* softmax-and-accumulate step shared by all bootstrap loops, src/jpmatLogBoot.cpp:264-269 (and :33-38):
 * per gene column: subtract max, exp, divide by (sum * scale), add into jp. */
static void softmax_accumulate(double *tjp, double *jp, int K, int ngenes, double scale) {
    for (int g = 0; g < ngenes; g++) {
        double *col = tjp + (size_t)g * K;
        double m = col[0];
        for (int k = 1; k < K; k++)
            if (col[k] > m) m = col[k];
        for (int k = 0; k < K; k++) col[k] = exp(col[k] - m);
        double s = arma_accumulate(col, K); /* sum(tjp, 0) */
        s *= scale;
        double *out = jp + (size_t)g * K;
        for (int k = 0; k < K; k++) out[k] += col[k] / s;
    }
}

/* gather outputs for returnpost 1..3, src/jpmatLogBoot.cpp:277-328 */
static void emit_individual(const table_t *t, const int *uci, int ngenes, const double *mag, int returnpost,
                            double *modes, double *post) {
    int K = t->K, ncells = t->ncells;
    if ((returnpost == 1 || returnpost == 3) && modes)
        for (int i = 0; i < ncells; i++)
            for (int j = 0; j < ngenes; j++) modes[(size_t)i * ngenes + j] = mag[t->maxi[i][uci[(size_t)i * ngenes + j]]];
    if ((returnpost == 2 || returnpost == 3) && post)
        for (int i = 0; i < ncells; i++) { /* post: ncells matrices, each G x K column-major */
            double *pl = post + (size_t)i * ngenes * K;
            for (int j = 0; j < ngenes; j++) {
                const double *col = t->pm[i] + (size_t)uci[(size_t)i * ngenes + j] * K;
                for (int k = 0; k < K; k++) pl[(size_t)k * ngenes + j] = col[k];
            }
        }
}

/*
 * logBootPosterior (src/jpmatLogBoot.cpp:100-331).
 *   models  ncells x 12 column-major (absent columns may hold NaN), ucl_flat/ucl_off the unique-count lists,
 *   uci     ngenes x ncells column-major 0-based indices into the lists, mag[K] natural-log magnitudes,
 *   boot_idx optional (nboot x ncells, draw order); NULL = generate with srand(seed)/rand() as the reference.
 * Outputs: jp ngenes x K column-major; modes ngenes x ncells; post ncells x (ngenes x K).
 */
int orc_log_boot_posterior(const double *models, int ncells, const int *ucl_flat, const int *ucl_off, const int *uci,
                           int ngenes, const double *mag, int K, int nboot, int seed, const int *boot_idx,
                           int returnpost, int localtheta, int sqlogit, int ensemble, double *jp, double *modes,
                           double *post) {
    table_t t;
    table_build(&t, models, ncells, ucl_flat, ucl_off, mag, K, localtheta, sqlogit, returnpost == 1 || returnpost == 3);
    double *jpt = (double *)calloc((size_t)K * ngenes, sizeof(double)); /* K x G, :217 */
    double *tjp = (double *)malloc(sizeof(double) * (size_t)K * ngenes);
    srand((unsigned)seed); /* :221 */
    if (ensemble) {        /* :224-237 */
        for (int j = 0; j < ncells; j++) {
            int nc = ucl_off[j + 1] - ucl_off[j];
            double *cp = (double *)malloc(sizeof(double) * (size_t)K * (nc > 0 ? nc : 1));
            for (int u = 0; u < nc; u++) {
                for (int k = 0; k < K; k++) cp[(size_t)u * K + k] = exp(t.pm[j][(size_t)u * K + k]);
                const double s = arma_accumulate(cp + (size_t)u * K, K); /* sum(cellucpost, 0) */
                for (int k = 0; k < K; k++) cp[(size_t)u * K + k] /= s;
            }
            for (int g = 0; g < ngenes; g++) {
                const double *col = cp + (size_t)uci[(size_t)j * ngenes + g] * K;
                for (int k = 0; k < K; k++) jpt[(size_t)g * K + k] += col[k];
            }
            free(cp);
        }
        for (int g = 0; g < ngenes; g++) {
            const double s = arma_accumulate(jpt + (size_t)g * K, K); /* sum(jp, 0) */
            for (int k = 0; k < K; k++) jpt[(size_t)g * K + k] /= s;
        }
    } else if (nboot == 0) { /* :239-249 */
        for (int j = 0; j < ncells; j++)
            for (int g = 0; g < ngenes; g++) {
                const double *col = t.pm[j] + (size_t)uci[(size_t)j * ngenes + g] * K;
                for (int k = 0; k < K; k++) jpt[(size_t)g * K + k] += col[k];
            }
        memcpy(tjp, jpt, sizeof(double) * (size_t)K * ngenes);
        memset(jpt, 0, sizeof(double) * (size_t)K * ngenes);
        softmax_accumulate(tjp, jpt, K, ngenes, 1.0);
    } else { /* :251-271 */
        for (int b = 0; b < nboot; b++) {
            memset(tjp, 0, sizeof(double) * (size_t)K * ngenes);
            for (int j = 0; j < ncells; j++) {
                int rj;
                if (boot_idx) {
                    rj = boot_idx[(size_t)b * ncells + j];
                } else {
                    while (ncells <= (rj = rand() / (RAND_MAX / ncells)))
                        ;
                }
                const double *pm = t.pm[rj];
                const int *ci = uci + (size_t)rj * ngenes;
                for (int g = 0; g < ngenes; g++) {
                    const double *col = pm + (size_t)ci[g] * K;
                    double *dst = tjp + (size_t)g * K;
                    for (int k = 0; k < K; k++) dst[k] += col[k];
                }
            }
            softmax_accumulate(tjp, jpt, K, ngenes, (double)nboot);
        }
    }
    for (int g = 0; g < ngenes; g++) /* :275 transpose */
        for (int k = 0; k < K; k++) jp[(size_t)k * ngenes + g] = jpt[(size_t)g * K + k];
    emit_individual(&t, uci, ngenes, mag, returnpost, modes, post);
    free(jpt);
    free(tjp);
    table_free(&t);
    return 0;
}

/*
 * logBootBatchPosterior (src/jpmatLogBoot.cpp:343-531).  boot_idx optional: nboot x D global cell ids,
 * D = sum(comp); NULL = draw with srand(seed)/rand() per the reference.  Note the reference fills `modes`
 * only for returnpost == 1 (:441,455) and has no returnpost == 3 branch; it also has no nboot == 0 branch.
 */
int orc_log_boot_batch_posterior(const double *models, int ncells, const int *ucl_flat, const int *ucl_off,
                                 const int *uci, int ngenes, const double *mag, int K, int nlevels,
                                 const int *pool_off, const int *pool_cells, const int *comp, int nboot, int seed,
                                 const int *boot_idx, int returnpost, int localtheta, int sqlogit, double *jp,
                                 double *modes, double *post) {
    table_t t;
    table_build(&t, models, ncells, ucl_flat, ucl_off, mag, K, localtheta, sqlogit, returnpost == 1);
    double *jpt = (double *)calloc((size_t)K * ngenes, sizeof(double));
    double *tjp = (double *)malloc(sizeof(double) * (size_t)K * ngenes);
    int D = 0;
    for (int k = 0; k < nlevels; k++)
        if (comp[k] > 0) D += comp[k];
    srand((unsigned)seed); /* :467 */
    for (int b = 0; b < nboot; b++) {
        memset(tjp, 0, sizeof(double) * (size_t)K * ngenes);
        int d = 0;
        for (int k = 0; k < nlevels; k++) {
            int nsamp = comp[k];
            if (nsamp <= 0) continue;
            const int *bi = pool_cells + pool_off[k];
            int npool = pool_off[k + 1] - pool_off[k];
            for (int j = 0; j < nsamp; j++, d++) {
                int cell;
                if (boot_idx) {
                    cell = boot_idx[(size_t)b * D + d];
                } else {
                    int rj;
                    while (npool <= (rj = rand() / (RAND_MAX / npool)))
                        ;
                    cell = bi[rj];
                }
                const double *pm = t.pm[cell];
                const int *ci = uci + (size_t)cell * ngenes;
                for (int g = 0; g < ngenes; g++) {
                    const double *col = pm + (size_t)ci[g] * K;
                    double *dst = tjp + (size_t)g * K;
                    for (int kk = 0; kk < K; kk++) dst[kk] += col[kk];
                }
            }
        }
        softmax_accumulate(tjp, jpt, K, ngenes, (double)nboot);
    }
    for (int g = 0; g < ngenes; g++)
        for (int k = 0; k < K; k++) jp[(size_t)k * ngenes + g] = jpt[(size_t)g * K + k];
    emit_individual(&t, uci, ngenes, mag, returnpost == 3 ? 2 : returnpost, modes, post);
    free(jpt);
    free(tjp);
    table_free(&t);
    return 0;
}

/*
 * Legacy dense form, src/jpmatLogBoot.cpp:11-42: matl = nmat matrices, each nrows x ncols column-major and
 * stored back to back; softmax is over columns per row (:33-37); NOT divided by nboot.
 */
void orc_jpmat_log_boot(const double *matl, int nmat, int nrows, int ncols, int nboot, int seed, const int *boot_idx,
                        double *jp) {
    size_t sz = (size_t)nrows * ncols;
    double *tjp = (double *)malloc(sizeof(double) * sz);
    memset(jp, 0, sizeof(double) * sz);
    srand((unsigned)seed);
    for (int i = 0; i < nboot; i++) {
        memset(tjp, 0, sizeof(double) * sz);
        for (int j = 0; j < nmat; j++) {
            int rj;
            if (boot_idx) {
                rj = boot_idx[(size_t)i * nmat + j];
            } else {
                while (nmat <= (rj = rand() / (RAND_MAX / nmat)))
                    ;
            }
            const double *am = matl + sz * rj;
            for (size_t e = 0; e < sz; e++) tjp[e] += am[e];
        }
        for (int r = 0; r < nrows; r++) {
            double m = tjp[r];
            for (int c = 1; c < ncols; c++)
                if (tjp[(size_t)c * nrows + r] > m) m = tjp[(size_t)c * nrows + r];
            double s = 0;
            for (int c = 0; c < ncols; c++) {
                double e = exp(tjp[(size_t)c * nrows + r] - m);
                tjp[(size_t)c * nrows + r] = e;
                s += e;
            }
            for (int c = 0; c < ncols; c++) jp[(size_t)c * nrows + r] += tjp[(size_t)c * nrows + r] / s;
        }
    }
    free(tjp);
}

/* src/jpmatLogBoot.cpp:48-86: matl holds all pools' matrices back to back, pool k = matrices
 * pool_off[k]..pool_off[k+1]-1; boot_idx (optional) = nboot x sum(comp) indices into matl. */
void orc_jpmat_log_batch_boot(const double *matl, int nlevels, const int *pool_off, const int *comp, int nrows,
                              int ncols, int nboot, int seed, const int *boot_idx, double *jp) {
    size_t sz = (size_t)nrows * ncols;
    double *tjp = (double *)malloc(sizeof(double) * sz);
    memset(jp, 0, sizeof(double) * sz);
    int D = 0;
    for (int k = 0; k < nlevels; k++)
        if (comp[k] > 0) D += comp[k];
    srand((unsigned)seed);
    for (int i = 0; i < nboot; i++) {
        memset(tjp, 0, sizeof(double) * sz);
        int d = 0;
        for (int k = 0; k < nlevels; k++) {
            int nsamp = comp[k];
            if (nsamp <= 0) continue;
            int nmat = pool_off[k + 1] - pool_off[k];
            for (int j = 0; j < nsamp; j++, d++) {
                int mi;
                if (boot_idx) {
                    mi = boot_idx[(size_t)i * D + d];
                } else {
                    int rj;
                    while (nmat <= (rj = rand() / (RAND_MAX / nmat)))
                        ;
                    mi = pool_off[k] + rj;
                }
                const double *am = matl + sz * mi;
                for (size_t e = 0; e < sz; e++) tjp[e] += am[e];
            }
        }
        for (int r = 0; r < nrows; r++) {
            double m = tjp[r];
            for (int c = 1; c < ncols; c++)
                if (tjp[(size_t)c * nrows + r] > m) m = tjp[(size_t)c * nrows + r];
            double s = 0;
            for (int c = 0; c < ncols; c++) {
                double e = exp(tjp[(size_t)c * nrows + r] - m);
                tjp[(size_t)c * nrows + r] = e;
                s += e;
            }
            for (int c = 0; c < ncols; c++) jp[(size_t)c * nrows + r] += tjp[(size_t)c * nrows + r] / s;
        }
    }
    free(tjp);
}

/* ------------------------------------------------------------------------------------ */
/* matSlideMult, src/matSlideMult.cpp:5-23.  m1, m2: nrows x n column-major; out: nrows x (2n-1). */
void orc_mat_slide_mult(const double *m1, const double *m2, int nrows, int n, double *out) {
    /* left half :12-16: out col (n-i) = sum_j m1[, j] * m2[, i-1+j], j = 0..n-i, for i = n..2 */
    for (int i = n; i > 1; i--) {
        double *o = out + (size_t)(n - i) * nrows;
        for (int r = 0; r < nrows; r++) o[r] = 0;
        for (int j = 0; j <= n - i; j++) {
            const double *a = m1 + (size_t)j * nrows, *b = m2 + (size_t)(i - 1 + j) * nrows;
            for (int r = 0; r < nrows; r++) o[r] += a[r] * b[r];
        }
    }
    /* right half :18-21: out col (n-2+i) = sum_j m1[, i-1+j] * m2[, j], j = 0..n-i, for i = 1..n */
    for (int i = 1; i <= n; i++) {
        double *o = out + (size_t)(n - 2 + i) * nrows;
        for (int r = 0; r < nrows; r++) o[r] = 0;
        for (int j = 0; j <= n - i; j++) {
            const double *a = m1 + (size_t)(i - 1 + j) * nrows, *b = m2 + (size_t)j * nrows;
            for (int r = 0; r < nrows; r++) o[r] += a[r] * b[r];
        }
    }
}

/* calculate.ratio.posterior, R/functions.R:3491-3510: optional column scaling by prior$y (:3494-3495),
 * matSlideMult (:3502), x/rowSums(x) (:3504; rowSums accumulates in long double).  out: G x (2K-1). */
void orc_ratio_posterior(const double *pmat1, const double *pmat2, int G, int K, const double *prior_y, double *out) {
    size_t sz = (size_t)G * K;
    double *a = (double *)malloc(sizeof(double) * sz), *b = (double *)malloc(sizeof(double) * sz);
    for (int k = 0; k < K; k++)
        for (int g = 0; g < G; g++) {
            size_t e = (size_t)k * G + g;
            a[e] = prior_y ? pmat1[e] * prior_y[k] : pmat1[e];
            b[e] = prior_y ? pmat2[e] * prior_y[k] : pmat2[e];
        }
    orc_mat_slide_mult(a, b, G, K, out);
    int n = 2 * K - 1;
    for (int g = 0; g < G; g++) {
        long double s = 0;
        for (int t = 0; t < n; t++) s += out[(size_t)t * G + g];
        double sd = (double)s;
        for (int t = 0; t < n; t++) out[(size_t)t * G + g] /= sd;
    }
    free(a);
    free(b);
}

/* get.ratio.posterior.Z.score, R/functions.R:3514-3531.  rpost: G x n column-major; zi: 1-based grid index
 * per gene (length G) or a single shared index (zi_len == 1). */
static void zscore(const double *rpost, int G, int n, const int *zi, int zi_len, double min_p, double *z) {
    for (int g = 0; g < G; g++) {
        long double rs = 0; /* rowSums of (rpost + min.p) */
        for (int t = 0; t < n; t++) rs += (rpost[(size_t)t * G + g] + min_p);
        double rsd = (double)rs;
        int z1 = zi_len == 1 ? zi[0] : zi[g];
        long double gsl = 0;
        /* rpost[, 1:(zi-1)]: for zi == 1 R's 1:0 selects column 1 (and the 0 is dropped) */
        int hi = (z1 - 1 >= 1) ? z1 - 1 : 1;
        for (int t = 0; t < hi; t++) gsl += (rpost[(size_t)t * G + g] + min_p) / rsd;
        double gs = (double)gsl;
        double zv = (rpost[(size_t)(z1 - 1) * G + g] + min_p) / rsd;
        double zl = fmin(0.0, orc_qnorm_upper(gs));
        double zg = fmax(0.0, orc_qnorm_upper(gs + zv));
        z[g] = (fabs(zl) > fabs(zg)) ? zl : zg;
    }
}

static int cmp_desc_idx(const void *a, const void *b, void *ctx) {
    const double *p = (const double *)ctx;
    int ia = *(const int *)a, ib = *(const int *)b;
    if (p[ia] > p[ib]) return -1;
    if (p[ia] < p[ib]) return 1;
    return (ia > ib) - (ia < ib); /* stable: R's order() is stable */
}

/* p.adjust(p, "BH"): pmin(1, cummin(n/i * p[o]))[ro], o = order(p, decreasing = TRUE), i = n:1 */
void orc_p_adjust_bh(const double *p, int n, double *out) {
    int *o = (int *)malloc(sizeof(int) * (n > 0 ? n : 1));
    for (int i = 0; i < n; i++) o[i] = i;
    qsort_r(o, n, sizeof(int), cmp_desc_idx, (void *)p);
    double cm = INFINITY;
    for (int r = 0; r < n; r++) {
        double v = (double)n / (double)(n - r) * p[o[r]];
        if (v < cm) cm = v;
        out[o[r]] = cm < 1 ? cm : 1;
    }
    free(o);
}

/*
 * quick.distribution.summary, R/functions.R:5039-5053.
 *   s_bdiffp G x n column-major, diffv[n] = as.numeric(colnames) (log10 fold-change grid),
 *   expectation: log2-scale H0 value(s), length 1 or G.
 * out: G x 6 column-major (lb, mle, ub, ce, Z, cZ); idx (optional): G x 3 column-major 0-based grid indices.
 */
void orc_distribution_summary(const double *s_bdiffp, int G, int n, const double *diffv, const double *expectation,
                              int exp_len, double *out, int *idx) {
    const double l2 = log10(2.0);
    double *z = (double *)malloc(sizeof(double) * (G > 0 ? G : 1));
    int *zi = (int *)malloc(sizeof(int) * (exp_len > 0 ? exp_len : 1));
    for (int g = 0; g < G; g++) {
        int mle = 0;
        double mv = s_bdiffp[g];
        long double cs = 0;
        int lb = 1, ub = n; /* 1-based; max(c(1, which(p<0.025))), min(c(n, which(p>0.975))) */
        int ub_set = 0;
        for (int t = 0; t < n; t++) {
            double v = s_bdiffp[(size_t)t * G + g];
            if (v > mv) { mv = v; mle = t; }
            cs += v;
            double c = (double)cs;
            if (c < 0.025 && t + 1 > lb) lb = t + 1;
            if (!ub_set && c > (1 - 0.025)) { ub = t + 1; ub_set = 1; }
        }
        double dlb = diffv[lb - 1] / l2, dmle = diffv[mle] / l2, dub = diffv[ub - 1] / l2;
        out[(size_t)0 * G + g] = dlb;
        out[(size_t)1 * G + g] = dmle;
        out[(size_t)2 * G + g] = dub;
        double cq = 0;
        if (dlb > 0) cq = dlb;
        if (dub < 0) cq = dub;
        out[(size_t)3 * G + g] = cq;
        if (idx) {
            idx[(size_t)0 * G + g] = lb - 1;
            idx[(size_t)1 * G + g] = mle;
            idx[(size_t)2 * G + g] = ub - 1;
        }
    }
    /* expectation/log2(10) -> nearest grid position, which.min(abs(mvs - x)) = first minimum */
    for (int e = 0; e < exp_len; e++) {
        double x = expectation[e] / log2(10.0);
        int bi = 0;
        double bv = fabs(diffv[0] - x);
        for (int t = 1; t < n; t++) {
            double d = fabs(diffv[t] - x);
            if (d < bv) { bv = d; bi = t; }
        }
        zi[e] = bi + 1;
    }
    zscore(s_bdiffp, G, n, zi, exp_len, 1e-15, z);
    double *pv = (double *)malloc(sizeof(double) * (G > 0 ? G : 1)), *pa = (double *)malloc(sizeof(double) * (G > 0 ? G : 1));
    for (int g = 0; g < G; g++) pv[g] = orc_pnorm_upper(fabs(z[g]));
    orc_p_adjust_bh(pv, G, pa);
    for (int g = 0; g < G; g++) {
        double sgn = (z[g] > 0) - (z[g] < 0);
        out[(size_t)4 * G + g] = z[g];
        out[(size_t)5 * G + g] = sgn * orc_qnorm_upper(pa[g]);
    }
    free(z);
    free(zi);
    free(pv);
    free(pa);
}

/* scde.expression.magnitude, R/functions.R:694-697: (log(counts) - corr.b) / corr.a; G x C column-major */
void orc_expression_magnitude(const int *counts, int G, int C, const double *corr_b, const double *corr_a, double *out) {
    for (int c = 0; c < C; c++)
        for (int g = 0; g < G; g++) {
            size_t e = (size_t)c * G + g;
            out[e] = (log((double)counts[e]) - corr_b[c]) / corr_a[c];
        }
}

/* ------------------------------------------------------------------------------------ */
/* host prep as scde.posteriors does it, R/functions.R:631-632: per cell unique() (first-appearance order)
 * and match()-1.  counts: G x C column-major.  ucl_flat must hold G*C ints (worst case). */
void orc_unique_counts(const int *counts, int G, int C, int *ucl_flat, int *ucl_off, int *uci) {
    int off = 0;
    ucl_off[0] = 0;
    /* open-addressing map value -> position */
    int cap = 1;
    while (cap < 2 * G + 2) cap <<= 1;
    int *keys = (int *)malloc(sizeof(int) * cap), *vals = (int *)malloc(sizeof(int) * cap);
    for (int c = 0; c < C; c++) {
        memset(vals, 0xff, sizeof(int) * cap);
        int nu = 0;
        for (int g = 0; g < G; g++) {
            int x = counts[(size_t)c * G + g];
            uint32_t h = ((uint32_t)x * 2654435761u) & (uint32_t)(cap - 1);
            while (vals[h] != -1 && keys[h] != x) h = (h + 1) & (uint32_t)(cap - 1);
            if (vals[h] == -1) {
                keys[h] = x;
                vals[h] = nu;
                ucl_flat[off + nu] = x;
                nu++;
            }
            uci[(size_t)c * G + g] = vals[h];
        }
        off += nu;
        ucl_off[c + 1] = off;
    }
    free(keys);
    free(vals);
}

/* ------------------------------------------------------------------------------------ */
/* CPU arm for bench.py: gene-chunked run of the joint posterior over `nthreads` workers, the way
 * scde.posteriors chunks genes over n.cores (R/functions.R:606-617): every chunk rebuilds its own unique-count
 * lists and lp table and then runs the bootstrap loop (the reference forks one process per chunk; plain
 * pthreads here -- the image has no libgomp).  All chunks use the same boot_idx (the n.cores = 1 semantics,
 * SURVEY.md section 8(e)).  counts: G x C column-major; boot_idx: nboot x D cell ids; jp: G x K column-major;
 * times (optional): seconds of the slowest worker in the table build and in the bootstrap loop. */
#include <pthread.h>
#include <time.h>
#include <unistd.h>

static double now_s(void) {
    struct timespec ts;
    clock_gettime(CLOCK_MONOTONIC, &ts);
    return ts.tv_sec + 1e-9 * ts.tv_nsec;
}

typedef struct {
    const double *models;
    const int *counts;
    const double *mag;
    const int *boot_idx;
    double *jp;
    int ncells, ngenes, K, nboot, D, g0, g1;
    double t_table, t_boot; /* seconds spent building the chunk's lp table / in the bootstrap loop */
} chunk_job_t;

static void *chunk_worker(void *arg) {
    chunk_job_t *jb = (chunk_job_t *)arg;
    int ng = jb->g1 - jb->g0, ncells = jb->ncells, K = jb->K, ngenes = jb->ngenes;
    if (ng <= 0) return NULL;
    int *sub = (int *)malloc(sizeof(int) * (size_t)ng * ncells);
    for (int c = 0; c < ncells; c++)
        memcpy(sub + (size_t)c * ng, jb->counts + (size_t)c * ngenes + jb->g0, sizeof(int) * ng);
    int *uf = (int *)malloc(sizeof(int) * (size_t)ng * ncells), *uo = (int *)malloc(sizeof(int) * (ncells + 1));
    int *ui = (int *)malloc(sizeof(int) * (size_t)ng * ncells);
    double t0 = now_s();
    orc_unique_counts(sub, ng, ncells, uf, uo, ui);
    table_t t;
    table_build(&t, jb->models, ncells, uf, uo, jb->mag, K, 0, 0, 0);
    double t1 = now_s();
    double *jpt = (double *)calloc((size_t)K * ng, sizeof(double));
    double *tjp = (double *)malloc(sizeof(double) * (size_t)K * ng);
    for (int b = 0; b < jb->nboot; b++) {
        memset(tjp, 0, sizeof(double) * (size_t)K * ng);
        for (int j = 0; j < jb->D; j++) {
            int rj = jb->boot_idx[(size_t)b * jb->D + j];
            const double *pm = t.pm[rj];
            const int *ci = ui + (size_t)rj * ng;
            for (int g = 0; g < ng; g++) {
                const double *col = pm + (size_t)ci[g] * K;
                double *dst = tjp + (size_t)g * K;
                for (int k = 0; k < K; k++) dst[k] += col[k];
            }
        }
        softmax_accumulate(tjp, jpt, K, ng, (double)jb->nboot);
    }
    for (int g = 0; g < ng; g++)
        for (int k = 0; k < K; k++) jb->jp[(size_t)k * ngenes + jb->g0 + g] = jpt[(size_t)g * K + k];
    jb->t_table = t1 - t0;
    jb->t_boot = now_s() - t1;
    free(jpt);
    free(tjp);
    table_free(&t);
    free(sub);
    free(uf);
    free(uo);
    free(ui);
    return NULL;
}

int orc_posteriors_chunked(const double *models, int ncells, const int *counts, int ngenes, const double *mag, int K,
                           int nboot, const int *boot_idx, int D, int nthreads, double *jp, double *times) {
    if (nthreads < 1) nthreads = 1;
    if (nthreads > ngenes) nthreads = ngenes > 0 ? ngenes : 1;
    pthread_t *th = (pthread_t *)malloc(sizeof(pthread_t) * nthreads);
    int *started = (int *)calloc(nthreads, sizeof(int));
    chunk_job_t *jobs = (chunk_job_t *)malloc(sizeof(chunk_job_t) * nthreads);
    for (int w = 0; w < nthreads; w++) {
        chunk_job_t jb = {models, counts, mag, boot_idx, jp, ncells, ngenes, K, nboot, D,
                          (int)((long long)ngenes * w / nthreads), (int)((long long)ngenes * (w + 1) / nthreads), 0, 0};
        jobs[w] = jb;
        if (pthread_create(&th[w], NULL, chunk_worker, &jobs[w]) == 0)
            started[w] = 1;
        else
            chunk_worker(&jobs[w]);
    }
    for (int w = 0; w < nthreads; w++)
        if (started[w]) pthread_join(th[w], NULL);
    if (times) { /* slowest worker: [0] table build, [1] bootstrap loop */
        times[0] = times[1] = 0;
        for (int w = 0; w < nthreads; w++) {
            if (jobs[w].t_table > times[0]) times[0] = jobs[w].t_table;
            if (jobs[w].t_boot > times[1]) times[1] = jobs[w].t_boot;
        }
    }
    free(th);
    free(started);
    free(jobs);
    return 0;
}

int orc_max_threads(void) {
    long n = sysconf(_SC_NPROCESSORS_ONLN);
    return n > 0 ? (int)n : 1;
}

/* ------------------------------------------------------------------------------------ */
/* scde.expression.prior (R/functions.R:225-254) and what it calls: scde.failure.probability (:725-750) and R's
 * stats::density.default (gaussian kernel, bw and weights given).  density.default is R code around two native
 * pieces -- BinDist (linear binning, src/library/stats/src/massdist.c) and fft() -- and approx(); R is not in
 * /root/reference, so this restates the published algorithm:
 *   n <- max(n, 512); if (n > 512) n <- 2^ceiling(log2(n));  lo <- from - 4 bw;  up <- to + 4 bw
 *   y <- BinDist(x, weights, lo, up, n)                       (2n values, the upper half zero)
 *   kords <- seq(0, 2 (up - lo), length.out = 2n);  kords[(n+2):(2n)] <- -kords[n:2];  kords <- dnorm(kords, sd = bw)
 *   kords <- fft(fft(y) * Conj(fft(kords)), inverse = TRUE);  kords <- pmax(0, Re(kords)[1:n] / length(y))
 *   approx(seq(lo, up, length.out = n), kords, seq(from, to, length.out = n.user))
 * The FFT here is a plain radix-2 transform (2n is a power of two); R's is Singleton's mixed-radix routine: equal up to
 * rounding (1e-16 of the largest value), which is why the tests compare the prior at 1e-12, not bit for bit. */
static void fft_radix2(double *re, double *im, int n, int inverse) {
    for (int i = 1, j = 0; i < n; i++) { /* bit reversal */
        int bit = n >> 1;
        for (; j & bit; bit >>= 1) j ^= bit;
        j ^= bit;
        if (i < j) {
            double t = re[i]; re[i] = re[j]; re[j] = t;
            t = im[i]; im[i] = im[j]; im[j] = t;
        }
    }
    for (int len = 2; len <= n; len <<= 1) {
        const double ang = 2 * M_PI / len * (inverse ? 1 : -1); /* R: forward transform uses exp(-2 pi i jk/n) */
        for (int i = 0; i < n; i += len)
            for (int k = 0; k < len / 2; k++) {
                const double wr = cos(ang * k), wi = sin(ang * k);
                const int a = i + k, b = i + k + len / 2;
                const double xr = re[b] * wr - im[b] * wi, xi = re[b] * wi + im[b] * wr;
                re[b] = re[a] - xr; im[b] = im[a] - xi;
                re[a] += xr; im[a] += xi;
            }
    }
}

/* x, w: nx weighted points (non-finite x are skipped as BinDist does); xout, yout: n_user values */
void orc_density_gaussian(const double *x, const double *w, long nx, double bw, int n_user, double from, double to,
                          double *xout, double *yout) {
    int n = n_user > 512 ? n_user : 512;
    if (n > 512) {
        int p = 1;
        while (p < n) p <<= 1;
        n = p;
    }
    const double lo = from - 4 * bw, up = to + 4 * bw;
    const int n2 = 2 * n;
    double *y = (double *)calloc((size_t)n2 * 4, sizeof(double));
    double *yi = y + n2, *kr = yi + n2, *ki = kr + n2;
    const int ixmin = 0, ixmax = n - 2;
    const double xdelta = (up - lo) / (n - 1);
    for (long i = 0; i < nx; i++) { /* BinDist */
        if (!isfinite(x[i])) continue;
        const double xpos = (x[i] - lo) / xdelta;
        const int ix = (int)floor(xpos);
        const double fx = xpos - ix, wi = w[i];
        if (ixmin <= ix && ix <= ixmax) {
            y[ix] += wi * (1 - fx);
            y[ix + 1] += wi * fx;
        } else if (ix == -1)
            y[0] += wi * fx;
        else if (ix == ixmax + 1)
            y[ix] += wi * (1 - fx);
    }
    for (int i = 0; i < n2; i++) { /* seq.int(0, 2*(up-lo), length.out = 2n): from + i*by */
        kr[i] = 0 + i * ((2 * (up - lo) - 0) / (n2 - 1));
    }
    kr[n2 - 1] = 2 * (up - lo);
    for (int i = n + 1; i < n2; i++) kr[i] = -kr[n2 - i]; /* kords[(n+2):(2n)] <- -kords[n:2] */
    for (int i = 0; i < n2; i++) kr[i] = exp(-0.5 * (kr[i] / bw) * (kr[i] / bw)) / (bw * sqrt(2 * M_PI)); /* dnorm */
    fft_radix2(y, yi, n2, 0);
    fft_radix2(kr, ki, n2, 0);
    for (int i = 0; i < n2; i++) { /* fft(y) * Conj(fft(kords)) */
        const double a = y[i], b = yi[i], c = kr[i], d = -ki[i];
        y[i] = a * c - b * d;
        yi[i] = a * d + b * c;
    }
    fft_radix2(y, yi, n2, 1); /* R's inverse transform is unnormalised */
    for (int i = 0; i < n; i++) {
        const double v = y[i] / n2;
        kr[i] = v > 0 ? v : 0; /* pmax.int(0, Re(kords)[1:n] / length(y)) */
    }
    /* approx(xords, kords, xout): linear interpolation, xords = seq.int(lo, up, length.out = n) */
    const double xby = (up - lo) / (n - 1), oby = n_user > 1 ? (to - from) / (n_user - 1) : 0;
    for (int i = 0; i < n_user; i++) {
        const double xo = (i == n_user - 1 && n_user > 1) ? to : from + i * oby;
        xout[i] = xo;
        /* R's approx1: binary search for the interval, then v[i] + (v[j] - v[i]) * ((x - x[i]) / (x[j] - x[i])) */
        int a = 0, b = n - 1;
        if (xo < lo || xo > up) {
            yout[i] = NAN;
            continue;
        }
        while (a < b - 1) {
            const int m = (a + b) / 2;
            const double xm = (m == n - 1) ? up : lo + m * xby;
            if (xo < xm) b = m; else a = m;
        }
        const double xa = (a == n - 1) ? up : lo + a * xby, xb = (b == n - 1) ? up : lo + b * xby;
        if (xo == xb) yout[i] = kr[b];
        else if (xo == xa) yout[i] = kr[a];
        else yout[i] = kr[a] + (kr[b] - kr[a]) * ((xo - xa) / (xb - xa));
    }
    free(y);
}

static int cmp_double(const void *a, const void *b) {
    const double x = *(const double *)a, y = *(const double *)b;
    return (x > y) - (x < y);
}

/* scde.failure.probability with per-cell magnitudes (the matrix branch, R/functions.R:736-741); NaN -> 0 (:748) */
void orc_failure_probability(const double *mag, int G, int C, const double *conc_a, const double *conc_b,
                             const double *conc_a2, double *out) {
    for (int c = 0; c < C; c++)
        for (int g = 0; g < G; g++) {
            const size_t e = (size_t)c * G + g;
            double eta = mag[e] * conc_a[c];
            if (conc_a2) eta += mag[e] * mag[e] * conc_a2[c];
            eta += conc_b[c];
            double v = 1 / (exp(eta) + 1);
            if (isnan(v)) v = 0;
            out[e] = v;
        }
}

/* scde.expression.prior.  models: C x 12 column-major (conc.a2 used when has_a2); max_value NaN = NULL (use the
 * max.quantile quantile, type 7, of the finite magnitudes).  Outputs x, y, lp, gw: length_out + 1 values each. */
void orc_expression_prior(const int *counts, int G, int C, const double *models, int has_a2, int length_out,
                          double pseudo_count, double bw, double max_quantile, double max_value, double *x, double *y,
                          double *lp, double *gw) {
    const size_t N = (size_t)G * C;
    double *fpkm = (double *)malloc(sizeof(double) * N * 4); /* fpkm, then the mirrored points and weights */
    double *wts = fpkm + N, *xx = wts + N;                   /* xx: 2N points; ww aliases after */
    double *mag = (double *)malloc(sizeof(double) * N);
    orc_expression_magnitude(counts, G, C, models + (size_t)CORRB_I * C, models + (size_t)CORRA_I * C, mag); /* :226 */
    orc_failure_probability(mag, G, C, models + (size_t)CONCA_I * C, models + (size_t)CONCB_I * C,
                            has_a2 ? models + (size_t)CONCA2_I * C : NULL, wts); /* :227 */
    long double ws = 0; /* R's sum() accumulates in long double */
    for (size_t i = 0; i < N; i++) {
        fpkm[i] = log10(exp(mag[i]) + 1); /* :228 */
        wts[i] = 1 - wts[i];              /* :229 */
        ws += wts[i];
    }
    for (size_t i = 0; i < N; i++) wts[i] /= (double)ws; /* :230 */
    if (isnan(max_value)) { /* :233-236 quantile(x[x < Inf], p = max.quantile), type 7 */
        size_t m = 0;
        for (size_t i = 0; i < N; i++)
            if (fpkm[i] < INFINITY) mag[m++] = fpkm[i];
        qsort(mag, m, sizeof(double), cmp_double);
        const double index = 1 + (m - 1) * max_quantile, fuzz = 4 * DBL_EPSILON;
        const double lo = floor(index + fuzz), hi = ceil(index - fuzz);
        const double qlo = mag[(size_t)lo - 1], qhi = mag[(size_t)hi - 1];
        double h = index - lo;
        if (fabs(h) < fuzz) h = 0;
        max_value = (h == 0) ? qlo : (1 - h) * qlo + h * qhi;
    }
    free(mag);
    /* :237 density(c(-fpkm, fpkm), weights = c(wts/2, wts/2)) */
    double *x2 = (double *)malloc(sizeof(double) * N * 4);
    double *w2 = x2 + 2 * N;
    for (size_t i = 0; i < N; i++) {
        x2[i] = -1 * fpkm[i];
        x2[N + i] = fpkm[i];
        w2[i] = w2[N + i] = wts[i] / 2;
    }
    const int n_user = 2 * length_out + 1;
    double *dx = (double *)malloc(sizeof(double) * n_user * 2), *dy = dx + n_user;
    orc_density_gaussian(x2, w2, (long)(2 * N), bw, n_user, -1 * max_value, max_value, dx, dy);
    const int K = length_out + 1;
    long double ys = 0;
    for (int k = 0; k < K; k++) { /* :239-241 */
        x[k] = dx[length_out + k];
        double v = dy[length_out + k];
        if (isnan(v)) v = 0;
        y[k] = v + pseudo_count / G;
        ys += y[k];
    }
    for (int k = 0; k < K; k++) {
        y[k] /= (double)ys; /* :242 */
        lp[k] = log(y[k]);  /* :247 */
    }
    /* :250 grid.weight = diff(10^c(x[1], x + c(diff(x)/2, 0)) - 1) */
    double prev = pow(10.0, x[0]) - 1;
    for (int k = 0; k < K; k++) {
        const double edge = x[k] + (k < K - 1 ? (x[k + 1] - x[k]) / 2 : 0);
        const double cur = pow(10.0, edge) - 1;
        gw[k] = cur - prev;
        prev = cur;
    }
    free(x2);
    free(dx);
    free(fpkm);
    (void)xx;
}
