// ratio_summary.cu -- group-difference posterior and its summary, fused per gene.
//
//   calculate.ratio.posterior  R/functions.R:3491-3510  (prior weighting, matSlideMult, row normalisation)
//   matSlideMult               src/matSlideMult.cpp:5-23 (row-wise full cross-correlation, 2n-1 lags)
//   quick.distribution.summary R/functions.R:5039-5053  (argmax, 2.5% / 97.5% cumulative bounds)
//   get.ratio.posterior.Z.score R/functions.R:3514-3531 (+1e-15, renormalise, tail mass -> qnorm)
//
// One CTA per gene (and contrast, in a batched launch): both weighted posteriors sit in shared memory, every thread owns a few lags of the sliding
// product and sums them in ascending j with separately rounded multiply and add (so the 2n-1 raw values are
// bit-identical to the reference's loop on a CPU build without FMA contraction); the row never returns to HBM
// unless the caller asked for the posterior.  R accumulates rowSums / cumsum in 80-bit long double; the device
// uses double-double (two-sum) accumulation, which rounds to the same double except on exact ties.
// Roofline: 2 n^2 flops against 16 n bytes in, 32 bytes out (or 8 (2n-1) when the posterior is kept) per gene --
// compute-light and tiny; reported against HBM bandwidth.
#include "common.cuh"
#include <cmath>

namespace scde {
namespace {

constexpr int R_THREADS = 256;

struct dd {
    double hi, lo;
};
__device__ __forceinline__ dd two_sum(double a, double b) {
    double s = __dadd_rn(a, b);
    double bb = __dadd_rn(s, -a);
    double e = __dadd_rn(__dadd_rn(a, -__dadd_rn(s, -bb)), __dadd_rn(b, -bb));
    return {s, e};
}
__device__ __forceinline__ dd fast_two_sum(double a, double b) {  // |a| >= |b|
    double s = __dadd_rn(a, b);
    double e = __dadd_rn(b, -__dadd_rn(s, -a));
    return {s, e};
}
__device__ __forceinline__ dd dd_add(dd x, double y) {
    dd t = two_sum(x.hi, y);
    t.lo = __dadd_rn(t.lo, x.lo);
    return fast_two_sum(t.hi, t.lo);
}
__device__ __forceinline__ dd dd_add(dd x, dd y) {
    dd t = two_sum(x.hi, y.hi);
    t.lo = __dadd_rn(t.lo, __dadd_rn(x.lo, y.lo));
    return fast_two_sum(t.hi, t.lo);
}
__device__ __forceinline__ double dd_val(dd x) { return __dadd_rn(x.hi, x.lo); }

// block-wide double-double sum; every thread gets the total.  s_hi/s_lo: R_THREADS/32 doubles each.
__device__ dd block_sum_dd(dd v, double *s_hi, double *s_lo) {
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
        dd other = {__shfl_xor_sync(0xffffffffu, v.hi, o), __shfl_xor_sync(0xffffffffu, v.lo, o)};
        // xor pairs add in both orders; dd_add is commutative in its result for the (hi, lo) sums used here
        v = (lane & o) ? dd_add(other, v) : dd_add(v, other);
    }
    __syncthreads();
    if (lane == 0) {
        s_hi[warp] = v.hi;
        s_lo[warp] = v.lo;
    }
    __syncthreads();
    dd t = {s_hi[0], s_lo[0]};
    for (int w = 1; w < R_THREADS / 32; ++w) t = dd_add(t, dd{s_hi[w], s_lo[w]});
    return t;
}

// qnorm(p, lower.tail = FALSE): Wichura AS 241 (PPND16)
__device__ double d_qnorm_upper(double p) {
    if (isnan(p)) return p;
    if (p < 0 || p > 1) return nan("");
    if (p == 0) return INFINITY;
    if (p == 1) return -INFINITY;
    double p_ = 0.5 - p + 0.5;
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
    r = (q < 0) ? p_ : p;
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

__global__ void __launch_bounds__(R_THREADS) ratio_summary_kernel(const RatioArgs a) {
    extern __shared__ double sm[];
    const int n = a.n, nout = 2 * n - 1;
    __shared__ double s_hi[R_THREADS / 32], s_lo[R_THREADS / 32];
    __shared__ double s_bv[R_THREADS / 32];
    __shared__ int s_bi[R_THREADS / 32];
    __shared__ int s_cnt[2];
    __shared__ double s_chunk_hi[R_THREADS / 32], s_chunk_lo[R_THREADS / 32];
    const int64_t g = blockIdx.x;
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    // batched launch: blockIdx.y is the contrast, whose inputs and outputs come from the device table
    const double *p1 = a.p1, *p2 = a.p2;
    int32_t *idx = a.idx;
    double *zo = a.z, *post = a.post;
    if (a.contrasts) {
        const RatioContrast c = a.contrasts[blockIdx.y];
        p1 = c.p1;
        p2 = c.p2;
        idx = c.idx;
        zo = c.z;
        post = c.post;
    }

    // Staging.  The sliding product below gives FOUR ADJACENT lags to a thread, so that a loaded p1[j] serves four
    // products and the four p2 values it meets are a window sliding along p2 (one new load per j): two shared-memory
    // loads per four multiply-adds instead of eight.  Adjacent threads then walk p1 / p2 at a stride of four doubles,
    // which would be an eight-way bank conflict; both vectors are therefore stored de-interleaved, q[u][m] = p[4 m + u - off],
    // so that the threads of a warp read consecutive words of one sub-array.  Zero padding on both sides stands for
    // the out-of-range terms: a product with +0 adds +0, which leaves the (non-negative) partial sums bit-identical to
    // the reference's shorter loops.
    const int off2 = 8 + ((4 - ((n - 1) & 3)) & 3);  // p2 index shift: (j + n - 1 - 4 g + off2) % 4 == j % 4 for every group g
    const int M1 = (n + 11) >> 2, M2 = (n + off2 + 11) >> 2;
    double *q1 = sm, *q2 = sm + 4 * M1, *out = sm + 4 * M1 + 4 * M2;  // out: nout values
    for (int i = tid; i < 4 * M1 + 4 * M2; i += R_THREADS) sm[i] = 0.0;
    __syncthreads();
    for (int j = tid; j < n; j += R_THREADS) {
        double x = p1[g * a.ld + j], y = p2[g * a.ld + j];
        if (a.prior) {
            const double w = a.prior[j];
            x = __dmul_rn(x, w);
            y = __dmul_rn(y, w);
        }
        q1[(j & 3) * M1 + (j >> 2)] = x;
        q2[((j + off2) & 3) * M2 + ((j + off2) >> 2)] = y;
    }
    if (tid < 2) s_cnt[tid] = 0;
    __syncthreads();

    // sliding product: lag index L in [0, 2n-2]; out[L] = sum_j p1[j] p2[j + n-1-L] over the j where both exist, j
    // ascending, multiply and add rounded separately (src/matSlideMult.cpp:13-21).  Group gi = lags 4 gi .. 4 gi + 3; its
    // j range is [max(0, 4 gi - (n-1)) rounded down to a multiple of 4, min(n-1, 4 gi + 3)], walked four j per
    // iteration.  Short and long groups are paired (gi, gi + ceil(NG/2)) so that every thread does about the same
    // number of iterations.
    {
        const int NG = (nout + 3) >> 2, half = (NG + 1) >> 1;
        for (int t = tid; t < half; t += R_THREADS) {
#pragma unroll 1
            for (int which = 0; which < 2; ++which) {
                const int gi = t + which * half;
                if (gi >= NG) break;
                const int L0 = 4 * gi;
                int j0 = L0 - (n - 1);
                j0 = j0 > 0 ? (j0 & ~3) : 0;
                const int j1 = min(n - 1, L0 + 3);
                const int iters = (j1 - j0 + 4) >> 2;
                const int i2 = j0 + (n - 1) - L0 + off2;  // shifted p2 index met by lag L0 at j0: a multiple of 4, >= 5
                const double *a1 = q1 + (j0 >> 2), *b2 = q2 + (i2 >> 2);
                // window: p2 values met by lags L0 + 1, + 2, + 3 at j0 (shifted indices i2 - 1, - 2, - 3)
                double w1 = q2[3 * M2 + ((i2 - 4) >> 2)], w2 = q2[2 * M2 + ((i2 - 4) >> 2)], w3 = q2[1 * M2 + ((i2 - 4) >> 2)];
                double acc0 = 0.0, acc1 = 0.0, acc2 = 0.0, acc3 = 0.0;
                for (int it = 0; it < iters; ++it) {
#pragma unroll
                    for (int u = 0; u < 4; ++u) {
                        const double x = a1[u * M1 + it], y = b2[u * M2 + it];
                        acc0 = __dadd_rn(acc0, __dmul_rn(x, y));
                        acc1 = __dadd_rn(acc1, __dmul_rn(x, w1));
                        acc2 = __dadd_rn(acc2, __dmul_rn(x, w2));
                        acc3 = __dadd_rn(acc3, __dmul_rn(x, w3));
                        w3 = w2;
                        w2 = w1;
                        w1 = y;
                    }
                }
                const double r[4] = {acc0, acc1, acc2, acc3};
#pragma unroll
                for (int i = 0; i < 4; ++i)
                    if (L0 + i < nout) {
                        out[L0 + i] = r[i];
                        if (a.raw) a.raw[g * a.ld_post + L0 + i] = r[i];
                    }
            }
        }
    }
    __syncthreads();
    if (!idx && !zo && !post) return;

    // x / rowSums(x)
    dd part = {0.0, 0.0};
    for (int L = tid; L < nout; L += R_THREADS) part = dd_add(part, out[L]);
    const double rs = dd_val(block_sum_dd(part, s_hi, s_lo));
    __syncthreads();
    for (int L = tid; L < nout; L += R_THREADS) {
        double r = out[L] / rs;
        out[L] = r;
        if (post) post[g * a.ld_post + L] = r;
    }
    __syncthreads();

    // which.max: first maximum
    {
        double bv = -INFINITY;
        int bi = 0x7fffffff;
        for (int L = tid; L < nout; L += R_THREADS) {
            double v = out[L];
            if (bi == 0x7fffffff || v > bv) {
                bv = v;
                bi = L;
            }
        }
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) {
            double ov = __shfl_xor_sync(0xffffffffu, bv, o);
            int oi = __shfl_xor_sync(0xffffffffu, bi, o);
            if (oi != 0x7fffffff && (bi == 0x7fffffff || ov > bv || (ov == bv && oi < bi))) {
                bv = ov;
                bi = oi;
            }
        }
        if (lane == 0) {
            s_bv[warp] = bv;
            s_bi[warp] = bi;
        }
    }
    // cumsum in contiguous per-thread chunks, then an exclusive scan of the chunk totals
    const int chunk = (nout + R_THREADS - 1) / R_THREADS;
    const int c0 = tid * chunk, c1 = min(nout, c0 + chunk);
    dd run = {0.0, 0.0};
    for (int L = c0; L < c1; ++L) run = dd_add(run, out[L]);
    // exclusive scan of the chunk totals (double-double): shuffles within the warp, then the warps' totals in order.
    // (A serial sum over the lower threads' totals cost 128 double-double additions per thread on average -- more FP64
    // work than the sliding product itself.)
    dd incl = run;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
        const dd other = {__shfl_up_sync(0xffffffffu, incl.hi, o), __shfl_up_sync(0xffffffffu, incl.lo, o)};
        if (lane >= o) incl = dd_add(other, incl);
    }
    if (lane == 31) {
        s_chunk_hi[warp] = incl.hi;
        s_chunk_lo[warp] = incl.lo;
    }
    dd off = {__shfl_up_sync(0xffffffffu, incl.hi, 1), __shfl_up_sync(0xffffffffu, incl.lo, 1)};
    if (lane == 0) off = dd{0.0, 0.0};
    __syncthreads();
    {
        dd woff = {0.0, 0.0};
        for (int w = 0; w < warp; ++w) woff = dd_add(woff, dd{s_chunk_hi[w], s_chunk_lo[w]});
        off = dd_add(woff, off);
    }
    int n_lt = 0, n_le = 0;
    run = off;
    for (int L = c0; L < c1; ++L) {
        run = dd_add(run, out[L]);
        const double cs = dd_val(run);
        n_lt += (cs < 0.025);
        n_le += !(cs > (1 - 0.025));
    }
    atomicAdd(&s_cnt[0], n_lt);
    atomicAdd(&s_cnt[1], n_le);

    // Z score: (r + 1e-15) renormalised
    part = dd{0.0, 0.0};
    for (int L = tid; L < nout; L += R_THREADS) part = dd_add(part, out[L] + 1e-15);
    const double rs2 = dd_val(block_sum_dd(part, s_hi, s_lo));  // has __syncthreads inside
    int zi = a.zero_index ? (a.n_zero == 1 ? a.zero_index[0] : a.zero_index[g]) : n;  // 1-based
    if (zi < 1) zi = 1;
    if (zi > nout) zi = nout;
    const int hi = (zi - 1 >= 1) ? zi - 1 : 1;  // R: 1:(zi-1) with zi == 1 selects column 1
    part = dd{0.0, 0.0};
    for (int L = tid; L < hi; L += R_THREADS) part = dd_add(part, (out[L] + 1e-15) / rs2);
    const double gs = dd_val(block_sum_dd(part, s_hi, s_lo));
    if (tid == 0) {
        double bv = s_bv[0];
        int bi = s_bi[0];
        for (int w = 1; w < R_THREADS / 32; ++w) {
            if (s_bi[w] != 0x7fffffff && (bi == 0x7fffffff || s_bv[w] > bv || (s_bv[w] == bv && s_bi[w] < bi))) {
                bv = s_bv[w];
                bi = s_bi[w];
            }
        }
        const int lb1 = max(1, s_cnt[0]);           // 1-based
        const int ub1 = min(nout, s_cnt[1] + 1);    // first index with cs > 0.975, else nout
        if (idx) {
            idx[0 * (int64_t)a.n_genes + g] = lb1 - 1;
            idx[1 * (int64_t)a.n_genes + g] = bi;
            idx[2 * (int64_t)a.n_genes + g] = ub1 - 1;
        }
        if (zo) {
            const double zv = (out[zi - 1] + 1e-15) / rs2;
            const double zl = fmin(0.0, d_qnorm_upper(gs));
            const double zg = fmax(0.0, d_qnorm_upper(gs + zv));
            zo[g] = (fabs(zl) > fabs(zg)) ? zl : zg;
        }
    }
}

__global__ void magnitude_kernel(const int32_t *__restrict__ counts, int64_t n, int G, const double *__restrict__ corr_b,
                                 const double *__restrict__ corr_a, double *__restrict__ out) {
    for (int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; e < n; e += (int64_t)gridDim.x * blockDim.x) {
        int c = (int)(e / G);
        out[e] = (log((double)counts[e]) - corr_b[c]) / corr_a[c];
    }
}

}  // namespace

cudaError_t launch_ratio_summary(const RatioArgs &a, cudaStream_t st) {
    if (a.n_genes <= 0) return cudaSuccess;
    const int off2 = 8 + ((4 - ((a.n - 1) & 3)) & 3);
    size_t smem = sizeof(double) * ((size_t)4 * ((a.n + 11) >> 2) + 4 * ((a.n + off2 + 11) >> 2) + 2 * a.n - 1);
    if (smem > 48 * 1024) {
        cudaError_t e = cudaFuncSetAttribute(ratio_summary_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
        if (e != cudaSuccess) return e;
    }
    if (!a.contrasts) {
        ratio_summary_kernel<<<a.n_genes, R_THREADS, smem, st>>>(a);
        return cudaGetLastError();
    }
    for (int c0 = 0; c0 < a.n_contrasts; c0 += 65535) {  // gridDim.y limit
        RatioArgs b = a;
        b.contrasts = a.contrasts + c0;
        const int nc = a.n_contrasts - c0 < 65535 ? a.n_contrasts - c0 : 65535;
        ratio_summary_kernel<<<dim3((unsigned)a.n_genes, (unsigned)nc), R_THREADS, smem, st>>>(b);
        cudaError_t e = cudaGetLastError();
        if (e != cudaSuccess) return e;
    }
    return cudaSuccess;
}

cudaError_t launch_magnitude(const int32_t *counts, int64_t n, int G, const double *corr_b, const double *corr_a,
                             double *out, cudaStream_t st) {
    if (n <= 0) return cudaSuccess;
    int64_t blocks = (n + 255) / 256;
    if (blocks > 148 * 16) blocks = 148 * 16;
    magnitude_kernel<<<(unsigned)blocks, 256, 0, st>>>(counts, n, G, corr_b, corr_a, out);
    return cudaGetLastError();
}

}  // namespace scde
