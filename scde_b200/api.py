"""Host-side mirror of scde's R API for the differential-expression posterior path.

Same function names (dots -> underscores), argument meaning and error behaviour as the reference:

    scde_expression_difference  <-  scde.expression.difference   R/functions.R:304-408
    scde_posteriors             <-  scde.posteriors              R/functions.R:566-670
    scde_expression_magnitude   <-  scde.expression.magnitude    R/functions.R:694-697
    calculate_ratio_posterior   <-  calculate.ratio.posterior    R/functions.R:3491-3510
    quick_distribution_summary  <-  quick.distribution.summary   R/functions.R:5039-5053
    mat_slide_mult / jpmat_log_boot / jpmat_log_batch_boot  <-  the R wrappers at R/functions.R:3534-3546

R data frames become pandas DataFrames (models: cells x coefficients; counts: genes x cells; prior: columns
``x`` and ``y``), factors become pandas Categoricals / Series.  All numeric work happens in libscde_b200.so
through the C ABI (``_lib``); this module only does what the R layer does: validation, reordering, packing,
labelling.  Nothing forks (SURVEY.md section 7).  ``n_cores`` is the reference's n.cores, which changes results: scde
splits the genes into n.cores chunks and draws every chunk's randomizations with its own Seed (R/functions.R:606-617).
By default (``chunked_draws=False``) ``n_cores`` is ignored and the results are those of ``n.cores = 1`` (Seed = 1, one
draw set for all genes).  ``chunked_draws=True`` honours it: ``scde_expression_difference`` and
``DifferenceSession.contrasts`` compute every chunk's draw set in the same device launches (``draw_chunks`` of the C
ABI), and ``scde_posteriors`` calls the library once per chunk, as the reference does.
"""
from __future__ import annotations

import ctypes as C
import sys
from typing import Optional, Sequence

import numpy as np
import pandas as pd

from . import _lib
from ._lib import check, f64, i32, lib, p_f64, p_i32

MODEL_COLUMNS = ["conc.b", "conc.a", "fail.r", "corr.b", "corr.a", "corr.theta", "corr.ltheta.b", "corr.ltheta.t",
                 "corr.ltheta.m", "corr.ltheta.s", "corr.ltheta.r", "conc.a2"]
MIN_SLOPE = 1e-10  # R/functions.R:579


def _stop(msg: str):
    raise ValueError("ERROR: " + msg)


def draw_chunk_ranges(G: int, n_cores: int) -> list:
    """The gene chunks of scde.posteriors with n.cores = n_cores (R/functions.R:606-617): the 0-based ranges [b, e) of
    split(seq_len(G), sort(rep_len(1:n, G))) when n > 1 and G > n (the first G %% n chunks one gene longer), else
    [(0, G)].  Chunk [b, e) draws with Seed = seed + b."""
    n = int(n_cores)
    if not (n > 1 and G > n):
        return [(0, G)]
    base, rem = divmod(G, n)
    out, b = [], 0
    for i in range(n):
        e = b + base + (1 if i < rem else 0)
        out.append((b, e))
        b = e
    return out


def _draw_chunks(chunked_draws: bool, n_cores: int, boot_idx) -> int:
    """draw_chunks of the C ABI for (chunked_draws, n_cores); explicit draws cannot be chunked."""
    if not chunked_draws:
        return 0
    if any(b is not None for b in (boot_idx if isinstance(boot_idx, (tuple, list)) else (boot_idx,))):
        raise ValueError("ERROR: chunked_draws draws every gene chunk from its own seed; it cannot be combined with boot_idx")
    if int(n_cores) < 1:
        raise ValueError("ERROR: n_cores must be >= 1")
    return int(n_cores)


# ------------------------------------------------------------------------------------------------
# small R idioms
def r_as_character_numeric(v: np.ndarray) -> np.ndarray:
    """as.numeric(as.character(x)): R prints doubles with 15 significant digits (R/functions.R:3507,5040)."""
    return np.array([float("%.15g" % t) for t in np.asarray(v, dtype=np.float64)], dtype=np.float64)


def r_seq_length(lo: float, hi: float, n: int) -> np.ndarray:
    """seq(lo, hi, length = n) as seq.default evaluates it: c(from, from + (1:(n-2)) * by, to)."""
    if n == 1:
        return np.array([lo], dtype=np.float64)
    by = (hi - lo) / (n - 1)
    out = lo + np.arange(n, dtype=np.float64) * by
    out[0], out[-1] = lo, hi
    return out


def fold_change_grid(x: np.ndarray) -> np.ndarray:
    """as.numeric(colnames(calculate.ratio.posterior(...))), log10 scale (R/functions.R:3506-3507)."""
    x = np.asarray(x, dtype=np.float64)
    return r_as_character_numeric(r_seq_length(x[0] - x[-1], x[-1] - x[0], 2 * len(x) - 1))


def marginals_from_prior(prior) -> np.ndarray:
    """R/functions.R:575-577."""
    m = np.power(10.0, np.asarray(prior["x"], dtype=np.float64)) - 1.0
    m[m < 0] = 0
    with np.errstate(divide="ignore"):
        return np.log(m)


def pack_models(models: pd.DataFrame, clamp: bool = True):
    """12-column matrix with NaN for absent columns (R/functions.R:601-604) after the slope clamp (:579-583;
    clamp = False: the models as they are, for scde.expression.prior / scde.failure.probability, which do not clamp)."""
    models = models.copy()
    ca = np.asarray(models["corr.a"], dtype=np.float64)
    bad = (ca < MIN_SLOPE) & clamp
    if bad.any():
        sys.stdout.write("WARNING: the following cells have negatively-correlated or 0-slope fits:  "
                         + " ".join(map(str, models.index[bad])) + " . Setting slopes to 1e-10.\n")
        ca = ca.copy()
        ca[bad] = MIN_SLOPE
        models["corr.a"] = ca
    mm = np.full((len(models), 12), np.nan, dtype=np.float64, order="F")
    for j, name in enumerate(MODEL_COLUMNS):
        if name in models.columns:
            mm[:, j] = np.asarray(models[name], dtype=np.float64)
    return mm, int("corr.ltheta.b" in models.columns), int("conc.a2" in models.columns)


def _counts_for_models(models: pd.DataFrame, counts) -> tuple[np.ndarray, list]:
    """counts[, match(rownames(models), colnames(counts))] as an int32 Fortran matrix + gene names."""
    if isinstance(counts, pd.DataFrame):
        if not all(c in counts.columns for c in models.index):
            _stop("provided count data does not cover all of the cells specified in the model matrix")
        sub = counts.loc[:, list(models.index)]
        return i32(sub.to_numpy()), list(sub.index)
    arr = np.asarray(counts)
    if arr.ndim != 2 or arr.shape[1] != len(models):
        _stop("provided count data does not cover all of the cells specified in the model matrix")
    return i32(arr), [str(i + 1) for i in range(arr.shape[0])]


def _unique_index(counts: np.ndarray):
    """ucl / uci (R/functions.R:631-632).  Sorted order instead of first appearance -- unobservable."""
    G, Cn = counts.shape
    flat, off = [], np.zeros(Cn + 1, dtype=np.int32)
    uci = np.empty((G, Cn), dtype=np.int32, order="F")
    for c in range(Cn):
        u, inv = np.unique(counts[:, c], return_inverse=True)
        flat.append(u.astype(np.int32))
        uci[:, c] = inv
        off[c + 1] = off[c] + len(u)
    return (np.concatenate(flat) if flat else np.zeros(0, np.int32)), off, uci


def _levels(f) -> tuple[np.ndarray, list]:
    """integer codes (-1 = NA) and level names of an R-factor-like object."""
    if isinstance(f, pd.Series):
        f = f.values if isinstance(f.dtype, pd.CategoricalDtype) else pd.Categorical(f)
    if not isinstance(f, pd.Categorical):
        f = pd.Categorical(f)
    return np.asarray(f.codes, dtype=np.int32), list(f.categories)


def _named_factor(f, names: Sequence[str]):
    """Align a (possibly named) factor to `names`; unnamed factors are taken positionally as R does."""
    if isinstance(f, pd.Series) and not f.index.equals(pd.RangeIndex(len(f))):
        f = f.reindex(list(names))
    codes, lev = _levels(f)
    if len(codes) != len(names):
        _stop("factor length does not match the number of cells in the model matrix")
    return codes, lev


# ------------------------------------------------------------------------------------------------
def scde_expression_magnitude(models: pd.DataFrame, counts) -> pd.DataFrame:
    """(log(counts) - corr.b) / corr.a per cell; genes x cells (R/functions.R:694-697)."""
    cm, genes = _counts_for_models(models, counts)
    G, Cn = cm.shape
    out = np.empty((G, Cn), dtype=np.float64, order="F")
    ctx = _lib.default_context()
    check(lib().scde_b200_expression_magnitude(ctx.handle, p_i32(cm), G, Cn,
                                               p_f64(f64(models["corr.b"])), p_f64(f64(models["corr.a"])), p_f64(out)))
    return pd.DataFrame(out, index=genes, columns=list(models.index))


def scde_posteriors(models: pd.DataFrame, counts, prior, n_randomizations: int = 100, batch=None, composition=None,
                    return_individual_posteriors: bool = False, return_individual_posterior_modes: bool = False,
                    ensemble_posterior: bool = False, n_cores: int = 20, seed: int = 1, boot_idx=None, context=None,
                    chunked_draws: bool = False):
    """Joint posterior of the cells in `models` (scde.posteriors, R/functions.R:566-670).

    Returns a genes x K DataFrame (columns = as.character(exp(marginals))) or, with the return_individual_* flags,
    a dict with ``jp`` plus ``modes`` (genes x cells) and/or ``post`` (dict cell -> genes x K DataFrame).
    `seed` / `boot_idx` expose what the reference fixes at Seed = 1 for n.cores = 1.  chunked_draws: one call per gene
    chunk of ``n_cores`` (draw_chunk_ranges) with Seed = seed + the chunk's first gene, results stacked -- the
    reference's own loop.
    """
    if _draw_chunks(chunked_draws, n_cores, boot_idx) > 1:
        cm, genes = _counts_for_models(models, counts)
        chunks = draw_chunk_ranges(cm.shape[0], n_cores)
        if len(chunks) > 1:
            cdf = pd.DataFrame(cm, index=genes, columns=list(models.index))
            parts = [scde_posteriors(models, cdf.iloc[b:e], prior, n_randomizations, batch, composition,
                                     return_individual_posteriors, return_individual_posterior_modes, ensemble_posterior,
                                     1, seed + b, None, context) for b, e in chunks]
            if isinstance(parts[0], pd.DataFrame):
                return pd.concat(parts)
            out = {"jp": pd.concat([p["jp"] for p in parts])}
            if "modes" in parts[0]:
                out["modes"] = pd.concat([p["modes"] for p in parts])
            if "post" in parts[0]:
                out["post"] = {cell: pd.concat([p["post"][cell] for p in parts]) for cell in parts[0]["post"]}
            return out
    cm, genes = _counts_for_models(models, counts)
    pools = comp = None
    if batch is not None:
        if composition is None:
            _stop("group composition must be provided if the batch argument is passed")
        bcodes, blev = _named_factor(batch, models.index)
        pools = [np.nonzero(bcodes == l)[0].astype(np.int32) for l in range(len(blev))]
        if isinstance(composition, (pd.Series, dict)):
            comp = np.array([int(dict(composition).get(l, 0)) for l in blev], dtype=np.int32)
        else:
            comp = i32(composition)
            if len(comp) != len(blev):
                _stop("composition must have one entry per batch level")
    mag = marginals_from_prior(prior)
    mm, lt, sq = pack_models(models)
    postflag = 0
    if return_individual_posteriors:
        postflag = 3 if return_individual_posterior_modes else 2
    elif return_individual_posterior_modes:
        postflag = 1
    flat, off, uci = _unique_index(cm)
    G, Cn = cm.shape
    K = len(mag)
    jp = np.empty((G, K), dtype=np.float64, order="F")
    want_modes = postflag in (1, 3) if batch is None else postflag == 1
    want_post = postflag in (2, 3)
    modes = np.empty((G, Cn), dtype=np.float64, order="F") if want_modes else None
    post = np.empty((Cn, K, G), dtype=np.float64) if want_post else None
    bi = None if boot_idx is None else i32(boot_idx, order="C")
    ctx = context or _lib.default_context()
    if batch is None:
        check(lib().scde_b200_log_boot_posterior(
            ctx.handle, p_f64(mm), Cn, p_i32(flat), p_i32(off), p_i32(uci), G, p_f64(f64(mag)), K,
            int(n_randomizations), int(seed), p_i32(bi), postflag, lt, sq, int(bool(ensemble_posterior)),
            p_f64(jp), p_f64(modes), p_f64(post)))
    else:
        poff = np.zeros(len(pools) + 1, dtype=np.int32)
        for k, p in enumerate(pools):
            poff[k + 1] = poff[k] + len(p)
        pcells = np.concatenate(pools).astype(np.int32) if pools else np.zeros(0, np.int32)
        check(lib().scde_b200_log_boot_batch_posterior(
            ctx.handle, p_f64(mm), Cn, p_i32(flat), p_i32(off), p_i32(uci), G, p_f64(f64(mag)), K, len(pools),
            p_i32(poff), p_i32(pcells), p_i32(comp), int(n_randomizations), int(seed), p_i32(bi), postflag, lt, sq,
            p_f64(jp), p_f64(modes), p_f64(post)))
    with np.errstate(over="ignore"):
        cols = ["%.15g" % v for v in np.exp(mag)]
    jpd = pd.DataFrame(jp, index=genes, columns=cols)
    if postflag == 0:
        return jpd
    out = {"jp": jpd}
    if modes is not None:
        out["modes"] = pd.DataFrame(modes, index=genes, columns=list(models.index))
    if post is not None:
        out["post"] = {cell: pd.DataFrame(post[i].T, index=genes, columns=cols) for i, cell in enumerate(models.index)}
    return out


# ------------------------------------------------------------------------------------------------
def mat_slide_mult(m1, m2, context=None) -> np.ndarray:
    """matSlideMult (R/functions.R:3544, src/matSlideMult.cpp:5)."""
    a, b = f64(m1), f64(m2)
    if a.shape != b.shape or a.ndim != 2:
        _stop("matSlideMult needs two matrices of the same shape")
    G, n = a.shape
    out = np.empty((G, 2 * n - 1), dtype=np.float64, order="F")
    ctx = context or _lib.default_context()
    check(lib().scde_b200_mat_slide_mult(ctx.handle, p_f64(a), p_f64(b), G, n, p_f64(out)))
    return out


def jpmat_log_boot(matl, nboot: int, seed: int, boot_idx=None, context=None) -> np.ndarray:
    """jpmatLogBoot (R/functions.R:3534, src/jpmatLogBoot.cpp:11)."""
    nrows, ncols = np.asarray(matl[0]).shape
    stack = np.empty((len(matl), ncols, nrows), dtype=np.float64)
    for i, m in enumerate(matl):
        stack[i] = np.asarray(m, dtype=np.float64).T
    jp = np.empty((nrows, ncols), dtype=np.float64, order="F")
    bi = None if boot_idx is None else i32(boot_idx, order="C")
    ctx = context or _lib.default_context()
    check(lib().scde_b200_jpmat_log_boot(ctx.handle, p_f64(stack), len(matl), nrows, ncols, int(nboot), int(seed),
                                         p_i32(bi), p_f64(jp)))
    return jp


def jpmat_log_batch_boot(matll, comp, nboot: int, seed: int, boot_idx=None, context=None) -> np.ndarray:
    """jpmatLogBatchBoot (R/functions.R:3540, src/jpmatLogBoot.cpp:48)."""
    flat = [m for pool in matll for m in pool]
    off = np.zeros(len(matll) + 1, dtype=np.int32)
    for k, pool in enumerate(matll):
        off[k + 1] = off[k] + len(pool)
    nrows, ncols = np.asarray(flat[0]).shape
    stack = np.empty((len(flat), ncols, nrows), dtype=np.float64)
    for i, m in enumerate(flat):
        stack[i] = np.asarray(m, dtype=np.float64).T
    jp = np.empty((nrows, ncols), dtype=np.float64, order="F")
    bi = None if boot_idx is None else i32(boot_idx, order="C")
    ctx = context or _lib.default_context()
    check(lib().scde_b200_jpmat_log_batch_boot(ctx.handle, p_f64(stack), len(matll), p_i32(off), p_i32(i32(comp)), nrows,
                                               ncols, int(nboot), int(seed), p_i32(bi), p_f64(jp)))
    return jp


def fisher_test_p_value(table: np.ndarray) -> float:
    """Two-sided p-value of fisher.test (R/functions.R:339) for the groups x batch contingency table: the total
    probability, under fixed margins, of the tables that are not more probable than the observed one (R's relative
    tolerance 1e-7).  2 x 2 tables are summed here (hypergeometric); larger ones go to scipy's exact r x c routine."""
    from math import lgamma

    t = np.asarray(table, dtype=np.int64)
    t = t[t.sum(axis=1) > 0][:, t.sum(axis=0) > 0]
    if t.shape[0] < 2 or t.shape[1] < 2:
        return 1.0
    if t.shape == (2, 2):
        r1, r2, c1 = int(t[0].sum()), int(t[1].sum()), int(t[:, 0].sum())
        lo, hi = max(0, c1 - r2), min(r1, c1)

        def lchoose(n, k):
            return lgamma(n + 1) - lgamma(k + 1) - lgamma(n - k + 1)

        ks = np.arange(lo, hi + 1)
        lp = np.array([lchoose(r1, k) + lchoose(r2, c1 - k) - lchoose(r1 + r2, c1) for k in ks])
        p = np.exp(lp - lp.max())
        p /= p.sum()
        obs = p[int(t[0, 0]) - lo]
        return float(min(1.0, p[p <= obs * (1 + 1e-7)].sum()))
    from scipy.stats import fisher_exact

    return float(fisher_exact(t).pvalue)


def _zero_index(diffv: np.ndarray, expectation) -> np.ndarray:
    """which.min(abs(mvs - expectation/log2(10))), 1-based (R/functions.R:3519,3524,5050)."""
    ex = np.atleast_1d(np.asarray(expectation, dtype=np.float64)) / np.log2(10.0)
    return np.array([int(np.argmin(np.abs(diffv - e))) + 1 for e in ex], dtype=np.int32)


def _summary_frame(idx: np.ndarray, z: np.ndarray, diffv: np.ndarray, genes, cz: Optional[np.ndarray] = None):
    """lb / mle / ub / ce / Z / cZ data frame from grid indices (R/functions.R:5045-5052)."""
    dq = diffv[idx] / np.log10(2.0)  # G x 3
    cq = np.zeros(len(z))
    sel = dq[:, 0] > 0
    cq[sel] = dq[sel, 0]
    sel = dq[:, 2] < 0
    cq[sel] = dq[sel, 2]
    if cz is None:
        cz = np.empty_like(z)
        check(lib().scde_b200_bh_cz(p_f64(f64(z)), len(z), p_f64(cz)))
    return pd.DataFrame({"lb": dq[:, 0], "mle": dq[:, 1], "ub": dq[:, 2], "ce": cq, "Z": z, "cZ": cz}, index=genes)


def calculate_ratio_posterior(pmat1, pmat2, prior, n_cores: int = 15, skip_prior_adjustment: bool = False,
                              context=None) -> pd.DataFrame:
    """calculate.ratio.posterior (R/functions.R:3491-3510): genes x (2K-1), columns labelled by log10 ratio."""
    genes = list(pmat1.index) if isinstance(pmat1, pd.DataFrame) else None
    a, b = f64(np.asarray(pmat1)), f64(np.asarray(pmat2))
    G, n = a.shape
    x = np.asarray(prior["x"], dtype=np.float64)
    py = None if skip_prior_adjustment else f64(prior["y"])
    post = np.empty((G, 2 * n - 1), dtype=np.float64, order="F")
    zi = np.array([n], dtype=np.int32)
    ctx = context or _lib.default_context()
    check(lib().scde_b200_ratio_posterior_summary(ctx.handle, p_f64(a), p_f64(b), G, n, p_f64(py), p_i32(zi), 1,
                                                  None, None, p_f64(post)))
    rv = r_seq_length(x[0] - x[-1], x[-1] - x[0], 2 * n - 1)
    return pd.DataFrame(post, index=genes, columns=["%.15g" % v for v in rv])


def quick_distribution_summary(pmat1, pmat2, prior, expectation=0.0, skip_prior_adjustment: bool = False,
                               genes=None, context=None) -> pd.DataFrame:
    """calculate.ratio.posterior + quick.distribution.summary fused on the device (no dense posterior)."""
    if genes is None and isinstance(pmat1, pd.DataFrame):
        genes = list(pmat1.index)
    a, b = f64(np.asarray(pmat1)), f64(np.asarray(pmat2))
    G, n = a.shape
    diffv = fold_change_grid(np.asarray(prior["x"], dtype=np.float64))
    py = None if skip_prior_adjustment else f64(prior["y"])
    zi = _zero_index(diffv, expectation)
    if len(zi) not in (1, G):
        _stop("the expectation parameter must be either one number or a vector equal to the number of genes being tested")
    idx = np.empty((G, 3), dtype=np.int32, order="F")
    z = np.empty(G, dtype=np.float64)
    ctx = context or _lib.default_context()
    check(lib().scde_b200_ratio_posterior_summary(ctx.handle, p_f64(a), p_f64(b), G, n, p_f64(py), p_i32(zi), len(zi),
                                                  p_i32(idx), p_f64(z), None))
    return _summary_frame(idx, z, diffv, genes)


# ------------------------------------------------------------------------------------------------
def _diff_args(counts, mm, prior_x, prior_y, group_codes, n_boot, seed, batch_codes, n_batch_levels, zero_index,
               zero_index_adjusted, local_theta, sqlogit, boot_idx, gene_range, batch_mm=None, batch_local_theta=0,
               batch_sqlogit=0, draw_chunks=0):
    """scde_b200_diff_args for the C ABI; returns (args, the host arrays it points into, processed genes, K, has_batch)."""
    keep_alive = []

    def keep(a):
        keep_alive.append(a)
        return a

    counts = keep(i32(counts))
    G_all, Cn = counts.shape
    K = len(prior_x)
    a = _lib.DiffArgs()
    a.n_genes, a.n_cells, a.n_grid = G_all, Cn, K
    a.counts = p_i32(counts)
    a.models = p_f64(keep(f64(mm)))
    a.prior_x = p_f64(keep(f64(prior_x)))
    a.prior_y = p_f64(keep(f64(prior_y)))
    a.group = p_i32(keep(i32(group_codes)))
    has_batch = batch_codes is not None and n_batch_levels > 1
    a.batch = p_i32(keep(i32(batch_codes))) if batch_codes is not None else None
    a.n_batch_levels = int(n_batch_levels)
    a.n_boot, a.seed = int(n_boot), int(seed)
    for i in range(4):
        a.boot_idx[i] = p_i32(keep(i32(boot_idx[i], order="C"))) if boot_idx[i] is not None else None
    zi = keep(i32(zero_index if zero_index is not None else [K]))
    a.zero_index, a.n_zero = p_i32(zi), len(zi)
    zia = keep(i32(zero_index_adjusted if zero_index_adjusted is not None else [2 * K - 1] * len(zi)))
    a.zero_index_adjusted = p_i32(zia)
    a.local_theta, a.square_logit_conc = int(local_theta), int(sqlogit)
    a.gene_begin, a.gene_end = int(gene_range[0]), int(gene_range[1])
    if batch_mm is not None:
        a.batch_models = p_f64(keep(f64(batch_mm)))
        a.batch_local_theta, a.batch_square_logit_conc = int(batch_local_theta), int(batch_sqlogit)
    a.draw_chunks = int(draw_chunks)
    G = (gene_range[1] - gene_range[0]) if tuple(gene_range) != (0, 0) else G_all
    return a, keep_alive, G, K, has_batch


def _diff_out(G, K, has_batch, want_posteriors, joint_posteriors, want_cz=False):
    """scde_b200_diff_out pointing into freshly allocated host arrays; returns (out, dict of those arrays)."""
    o = _lib.DiffOut()
    res = {"idx": np.empty((G, 3), np.int32, order="F"), "z": np.empty(G)}
    o.idx, o.z = p_i32(res["idx"]), p_f64(res["z"])
    if want_cz:  # BH-corrected cZ over the genes of the call (scde_b200_expression_difference only)
        res["cz"] = np.empty(G)
        o.cz = p_f64(res["cz"])
    if has_batch:
        for k in ("batch", "adjusted"):
            res[k + "_idx"] = np.empty((G, 3), np.int32, order="F")
            res[k + "_z"] = np.empty(G)
            if want_cz:
                res[k + "_cz"] = np.empty(G)
        o.batch_idx, o.batch_z = p_i32(res["batch_idx"]), p_f64(res["batch_z"])
        o.adjusted_idx, o.adjusted_z = p_i32(res["adjusted_idx"]), p_f64(res["adjusted_z"])
        if want_cz:
            o.batch_cz, o.adjusted_cz = p_f64(res["batch_cz"]), p_f64(res["adjusted_cz"])
    if want_posteriors:
        res["difference_posterior"] = np.empty((G, 2 * K - 1), order="F")
        o.difference_posterior = p_f64(res["difference_posterior"])
        if has_batch:
            res["batch_difference_posterior"] = np.empty((G, 2 * K - 1), order="F")
            res["adjusted_difference_posterior"] = np.empty((G, 4 * K - 3), order="F")
            o.batch_difference_posterior = p_f64(res["batch_difference_posterior"])
            o.adjusted_difference_posterior = p_f64(res["adjusted_difference_posterior"])
    if joint_posteriors or want_posteriors:
        res["joint_posteriors"] = [np.empty((G, K), order="F") for _ in range(2)]
        for i in range(2):
            o.joint_posteriors[i] = p_f64(res["joint_posteriors"][i])
        if has_batch:
            res["batch_joint_posteriors"] = [np.empty((G, K), order="F") for _ in range(2)]
            for i in range(2):
                o.batch_joint_posteriors[i] = p_f64(res["batch_joint_posteriors"][i])
    return o, res


def expression_difference_call(ctx: _lib.Context, counts: np.ndarray, mm: np.ndarray, prior_x, prior_y, group_codes,
                               n_boot: int, seed: int = 1, batch_codes=None, n_batch_levels: int = 0, zero_index=None,
                               zero_index_adjusted=None, local_theta: int = 0, sqlogit: int = 0, boot_idx=(None,) * 4,
                               gene_range=(0, 0), want_posteriors: bool = False, joint_posteriors: bool = False,
                               batch_mm=None, batch_local_theta: int = 0, batch_sqlogit: int = 0, n_cores: int = 1,
                               chunked_draws: bool = False):
    """The one-shot C-ABI call (scde_b200_expression_difference): host buffers in, host buffers out.  The count matrix is
    uploaded in cell chunks while the table rows of the chunks already on the device are being built.  chunked_draws:
    the draws of n.cores = n_cores (see the module docstring)."""
    dc = _draw_chunks(chunked_draws, n_cores, boot_idx)
    a, keep_alive, G, K, has_batch = _diff_args(counts, mm, prior_x, prior_y, group_codes, n_boot, seed, batch_codes,
                                                n_batch_levels, zero_index, zero_index_adjusted, local_theta, sqlogit,
                                                boot_idx, gene_range, batch_mm, batch_local_theta, batch_sqlogit, dc)
    o, res = _diff_out(G, K, has_batch, want_posteriors, joint_posteriors, want_cz=tuple(gene_range) == (0, 0))
    st = _lib.Stats()
    check(lib().scde_b200_expression_difference(ctx.handle, C.byref(a), C.byref(o), C.byref(st)))
    del keep_alive
    res["stats"] = st.as_dict()
    return res


class DifferenceJob:
    """Device-resident scde.expression.difference: upload once, run, download (C ABI split form)."""

    def __init__(self, ctx: _lib.Context, counts: np.ndarray, mm: np.ndarray, prior_x, prior_y, group_codes,
                 n_boot: int, seed: int = 1, batch_codes=None, n_batch_levels: int = 0, zero_index=None,
                 zero_index_adjusted=None, local_theta: int = 0, sqlogit: int = 0, boot_idx=(None,) * 4,
                 gene_range=(0, 0), want_posteriors: bool = False, batch_mm=None, batch_local_theta: int = 0,
                 batch_sqlogit: int = 0, n_cores: int = 1, chunked_draws: bool = False):
        self.ctx = ctx
        dc = _draw_chunks(chunked_draws, n_cores, boot_idx)
        a, keep_alive, self.G, self.K, self.has_batch = _diff_args(
            counts, mm, prior_x, prior_y, group_codes, n_boot, seed, batch_codes, n_batch_levels, zero_index,
            zero_index_adjusted, local_theta, sqlogit, boot_idx, gene_range, batch_mm, batch_local_theta, batch_sqlogit,
            dc)
        self.want_posteriors = bool(want_posteriors)
        self._job = C.c_void_p()
        check(lib().scde_b200_diff_upload(ctx.handle, C.byref(a), int(want_posteriors), C.byref(self._job)))
        del keep_alive  # the host arrays only had to outlive the upload call

    def run(self):
        """Queue all device work on the context stream (asynchronous)."""
        check(lib().scde_b200_diff_run(self.ctx.handle, self._job))

    def download(self, joint_posteriors: bool = False):
        o, res = _diff_out(self.G, self.K, self.has_batch, self.want_posteriors, joint_posteriors)
        st = _lib.Stats()
        check(lib().scde_b200_diff_download(self.ctx.handle, self._job, C.byref(o), C.byref(st)))
        res["stats"] = st.as_dict()
        return res

    def close(self):
        if self._job:
            lib().scde_b200_diff_free(self.ctx.handle, self._job)
            self._job = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


def _batch_model_matrix(models: pd.DataFrame, batch_models):
    """batch.models (R/functions.R:304,356), the error models of the composition-sampled joints, as the column-major
    matrix of the cells of `models` in their order: ``(matrix, local_theta, sqlogit)``, or ``(None, 0, 0)`` when they
    are `models` themselves or not given."""
    if batch_models is None or batch_models is models:
        return None, 0, 0
    if list(batch_models.index) != list(models.index):
        if not all(c in batch_models.index for c in models.index):
            _stop("batch.models does not cover all of the cells specified in the model matrix")
        batch_models = batch_models.loc[list(models.index)]
    return pack_models(batch_models)


def _zero_indices(x: np.ndarray, expectation, G: int):
    """The fold-change grid of the prior's grid `x`, the grid of the batch-adjusted difference, and the 1-based H0 index
    of `expectation` in each: ``diffv, zi, adiffv, zia``."""
    diffv = fold_change_grid(x)
    zi = _zero_index(diffv, expectation)
    if len(zi) not in (1, G):
        _stop("the expectation parameter must be either one number or a vector equal to the number of genes being tested")
    adiffv = fold_change_grid(diffv)
    return diffv, zi, adiffv, _zero_index(adiffv, expectation)


def _difference_result(r: dict, genes, diffv, adiffv, kcols, names, correct_batch: bool, return_posteriors: bool,
                       stats: dict):
    """What scde.expression.difference returns, from one contrast's arrays `r` (keys as from _diff_out; the two joint
    posteriors under ``joint_posteriors``, labelled `names`): the ``lb mle ub ce Z cZ`` frame with ``attrs["stats"]``,
    or the reference's list as a dict with batch correction and/or posteriors."""
    res = _summary_frame(r["idx"], r["z"], diffv, genes, cz=r.get("cz"))
    if not correct_batch and not return_posteriors:
        res.attrs["stats"] = stats
        return res
    out = {}
    if correct_batch:
        out["batch.adjusted"] = _summary_frame(r["adjusted_idx"], r["adjusted_z"], adiffv, genes, cz=r.get("adjusted_cz"))
    out["results"] = res
    if correct_batch:
        out["batch.effect"] = _summary_frame(r["batch_idx"], r["batch_z"], diffv, genes, cz=r.get("batch_cz"))
    if return_posteriors:
        out["difference.posterior"] = pd.DataFrame(r["difference_posterior"], index=genes,
                                                   columns=["%.15g" % v for v in diffv])
        out["joint.posteriors"] = {n: pd.DataFrame(jp, index=genes, columns=kcols)
                                   for n, jp in zip(names, r["joint_posteriors"])}
        if correct_batch:
            out["batch.adjusted.difference.posterior"] = pd.DataFrame(
                r["adjusted_difference_posterior"], index=genes, columns=["%.15g" % v for v in adiffv])
    out["stats"] = stats
    return out


def scde_expression_difference(models: pd.DataFrame, counts, prior, groups=None, batch=None,
                               n_randomizations: int = 150, n_cores: int = 10, batch_models=None,
                               return_posteriors: bool = False, expectation=0, verbose: int = 0, seed: int = 1,
                               context=None, boot_idx=(None,) * 4, chunked_draws: bool = False):
    """scde.expression.difference (R/functions.R:304-408).

    Returns the ``lb mle ub ce Z cZ`` data frame (genes as rows), or a dict shaped like the reference's list when
    `batch` and/or `return_posteriors` are given (keys: ``results``, ``batch.adjusted``, ``batch.effect``,
    ``difference.posterior``, ``batch.adjusted.difference.posterior``, ``joint.posteriors``).
    chunked_draws: honour n_cores as the reference's n.cores (one draw set per gene chunk; see the module docstring).
    """
    _draw_chunks(chunked_draws, n_cores, boot_idx)  # argument errors before any library call
    cm, genes = _counts_for_models(models, counts)
    if groups is None:
        groups = models.attrs.get("groups")
        if groups is None:
            _stop("groups factor is not provided, and models structure is lacking groups attribute")
        groups = pd.Categorical(groups)
    gcodes, glev = _named_factor(groups, models.index)
    if len(glev) != 2:
        _stop("wrong number of levels in the grouping factor (" + " ".join(map(str, glev)) + "), but must be two.")
    correct_batch = False
    bcodes, blev = None, []
    if batch is not None:
        bcodes, blev = _named_factor(batch, models.index)
        if len(blev) > 1:
            correct_batch = True
        elif verbose:
            sys.stdout.write("WARNING: only one batch level detected. Nothing to correct for.")
    bmm, blt, bsq = _batch_model_matrix(models, batch_models) if correct_batch else (None, 0, 0)
    if correct_batch:
        # check batch-group interactions (R/functions.R:336-349): table(groups, batch), fisher.test, warning below 1e-3
        bgti = pd.crosstab(pd.Series(np.asarray(gcodes), name="groups"), pd.Series(np.asarray(bcodes), name="batch"))
        bgti = bgti.loc[[i for i in bgti.index if i >= 0], [c for c in bgti.columns if c >= 0]]
        if verbose:
            sys.stdout.write("controlling for batch effects. interaction:\n")
            sys.stdout.write(str(bgti) + "\n")
        pval = fisher_test_p_value(bgti.to_numpy())
        if pval < 1e-3:
            sys.stdout.write("WARNING: strong interaction between groups and batches! Correction may be ineffective:\n")
            sys.stdout.write(f"Fisher's Exact Test for Count Data: p-value = {pval:.4g}\n")
    elif verbose:
        sys.stdout.write("comparing groups:\n")
        sys.stdout.write(str(pd.Series([glev[c] for c in gcodes if c >= 0]).value_counts().sort_index()) + "\n")
    mm, lt, sq = pack_models(models)
    x = np.asarray(prior["x"], dtype=np.float64)
    diffv, zi, adiffv, zia = _zero_indices(x, expectation, cm.shape[0])
    ctx = context or _lib.default_context()
    if verbose:
        sys.stdout.write("calculating difference posterior\n")
    res = expression_difference_call(ctx, cm, mm, x, np.asarray(prior["y"], dtype=np.float64), gcodes, n_randomizations, seed,
                                     batch_codes=bcodes if correct_batch else None,
                                     n_batch_levels=len(blev) if correct_batch else 0, zero_index=zi,
                                     zero_index_adjusted=zia, local_theta=lt, sqlogit=sq, boot_idx=boot_idx,
                                     want_posteriors=return_posteriors, batch_mm=bmm, batch_local_theta=blt,
                                     batch_sqlogit=bsq, n_cores=n_cores, chunked_draws=chunked_draws)
    if verbose:
        sys.stdout.write("summarizing differences\n")
    with np.errstate(over="ignore"):
        kcols = ["%.15g" % v for v in np.exp(marginals_from_prior(prior))]
    return _difference_result(res, genes, diffv, adiffv, kcols, glev, correct_batch, return_posteriors, res["stats"])


def scde_test_gene_expression_difference(gene, models: pd.DataFrame, counts: pd.DataFrame, prior, groups=None, batch=None,
                                         batch_models=None, n_randomizations: int = 1000, show_plots: bool = False,
                                         return_details: bool = False, verbose: bool = False, expectation=0,
                                         n_cores: int = 1, seed: int = 1, context=None):
    """Numeric core of scde.test.gene.expression.difference (R/functions.R:783-947; plotting is out of scope).

    One gene, n.randomizations = 1e3 by default, individual posteriors kept (`return.details`).  Goes through the same
    C-ABI entry points as the reference's R code does: two (or four) scde_posteriors calls, calculate.ratio.posterior,
    quick.distribution.summary.
    """
    if gene not in counts.index:
        _stop(f"specified gene ({gene}) is not found in the count data")
    if batch_models is None:
        batch_models = models
    sub = counts.loc[[gene], list(models.index)]
    if groups is None:
        groups = models.attrs.get("groups")
        if groups is None:
            _stop("groups factor is not provided, and models structure is lacking groups attribute")
        groups = pd.Categorical(groups)
    gcodes, glev = _named_factor(groups, models.index)
    if len(glev) != 2:
        _stop("wrong number of levels in the grouping factor (" + " ".join(map(str, glev)) + "), but must be two.")
    ctx = context or _lib.default_context()
    jpl = []
    for lev in range(2):
        ii = np.nonzero(gcodes == lev)[0]
        jpl.append(scde_posteriors(models.iloc[ii], sub.iloc[:, ii], prior, n_randomizations=n_randomizations,
                                   return_individual_posteriors=True, seed=seed, context=ctx))
    diffv = fold_change_grid(np.asarray(prior["x"], dtype=np.float64))
    bdiffp = calculate_ratio_posterior(jpl[0]["jp"], jpl[1]["jp"], prior, context=ctx)
    rep = quick_distribution_summary(jpl[0]["jp"], jpl[1]["jp"], prior, expectation=expectation, genes=[gene], context=ctx)
    correct_batch = False
    if batch is not None:
        bcodes, blev = _named_factor(batch, models.index)
        correct_batch = len(blev) > 1
    if correct_batch:
        bjpl = []
        for lev in range(2):
            ii = np.nonzero(gcodes == lev)[0]
            comp = np.bincount(bcodes[ii][bcodes[ii] >= 0], minlength=len(blev)).astype(np.int32)
            bjpl.append(scde_posteriors(batch_models, sub, prior, n_randomizations=n_randomizations, batch=batch,
                                        composition=comp, seed=seed, context=ctx))
        bb = calculate_ratio_posterior(bjpl[0], bjpl[1], prior, context=ctx)
        uni = {"x": diffv, "y": np.full(len(diffv), 1.0 / len(diffv))}
        abd = calculate_ratio_posterior(bdiffp, bb, uni, skip_prior_adjustment=True, context=ctx)
        arep = quick_distribution_summary(bdiffp, bb, uni, expectation=expectation, skip_prior_adjustment=True,
                                          genes=[gene], context=ctx)
        if return_details:
            return {"results": arep, "difference.posterior": abd, "results.nobatchcorrection": rep}
        return arep
    if return_details:
        return {"results": rep, "difference.posterior": bdiffp, "posteriors": {glev[i]: jpl[i] for i in range(2)}}
    return rep


# ------------------------------------------------------------------------------------------------
# many contrasts on one resident dataset
def _side_label(levels: Sequence) -> str:
    return str(levels[0]) if len(levels) == 1 else "+".join(str(v) for v in levels)


def expand_contrasts(levels: Sequence, contrasts="pairs") -> list:
    """The contrasts of a call as ``(label, levels of A, levels of B, name of A, name of B)``, A the first level of the
    two-level factor each contrast stands for (a positive fold change = higher in A).

    ``"pairs"``: every (a, b) with a before b in level order; ``"rest"``: every level against the union of the others,
    B named ``"rest"``; otherwise a list of (A, B), each side a level name or a list of level names (their union).
    The labels are ``"<A> vs <B>"`` with a union written ``a+b``.  Host only."""
    levels = list(levels)
    out = []
    if isinstance(contrasts, str):
        if contrasts not in ("pairs", "rest"):
            _stop(f'contrasts must be "pairs", "rest" or a list of pairs, not "{contrasts}"')
        if len(levels) < 2:
            _stop("the grouping factor needs at least two levels to compare")
        if contrasts == "pairs":
            for i, a in enumerate(levels):
                for b in levels[i + 1:]:
                    out.append((f"{a} vs {b}", [a], [b], str(a), str(b)))
        else:
            for a in levels:
                rest = [b for b in levels if b != a]
                out.append((f"{a} vs rest", [a], rest, str(a), "rest"))
        return out
    pairs = list(contrasts)
    if not pairs:
        _stop("no contrasts given")
    for pair in pairs:
        if isinstance(pair, str) or len(pair) != 2:
            _stop("each contrast must be a pair (A, B) of level names or lists of level names")
        sides = []
        for side in pair:
            lv = [side] if isinstance(side, str) or not isinstance(side, (list, tuple, set, np.ndarray)) else list(side)
            if not lv:
                _stop("a side of a contrast names no level")
            for v in lv:
                if v not in levels:
                    _stop(f"unknown level {v} in a contrast (levels: " + " ".join(map(str, levels)) + ")")
            if len(set(lv)) != len(lv):
                _stop("a side of a contrast names a level twice")
            sides.append(lv)
        if set(sides[0]) & set(sides[1]):
            _stop("the two sides of a contrast share level(s) " + " ".join(map(str, sorted(set(sides[0]) & set(sides[1]), key=str))))
        na, nb = _side_label(sides[0]), _side_label(sides[1])
        out.append((f"{na} vs {nb}", sides[0], sides[1], na, nb))
    labels = [c[0] for c in out]
    if len(set(labels)) != len(labels):
        _stop("a contrast is listed twice")
    return out


class DifferenceSession:
    """scde.expression.difference for many contrasts over one set of cells.

    The count matrix, its unique-count index and the log-posterior table of every cell stay on the device until
    ``close()``; each ``contrasts()`` call computes every named group's joint posterior once and all requested contrasts
    from them.  Every contrast equals ``scde_expression_difference`` called with the corresponding two-level factor (the
    cells of neither side NA).  While a session is open, the one-shot call on the same context is refused.
    """

    def __init__(self, models: pd.DataFrame, counts, prior, context=None):
        self.models = models
        cm, self.genes = _counts_for_models(models, counts)
        mm, self._lt, self._sq = pack_models(models)
        self._x = f64(np.asarray(prior["x"], dtype=np.float64))
        self._y = f64(np.asarray(prior["y"], dtype=np.float64))
        with np.errstate(over="ignore"):
            self._kcols = ["%.15g" % v for v in np.exp(marginals_from_prior(prior))]
        self.ctx = context or _lib.default_context()
        self.G, self.C, self.K = cm.shape[0], cm.shape[1], len(self._x)
        a = _lib.DatasetArgs()
        a.n_genes, a.n_cells, a.n_grid = self.G, self.C, self.K
        a.counts, a.models, a.prior_x, a.prior_y = p_i32(cm), p_f64(mm), p_f64(self._x), p_f64(self._y)
        a.local_theta, a.square_logit_conc = self._lt, self._sq
        self._ds = C.c_void_p()
        st = _lib.Stats()
        check(lib().scde_b200_dataset_create(self.ctx.handle, C.byref(a), C.byref(self._ds), C.byref(st)))
        self.create_stats = st.as_dict()
        self.last_stats = None

    def contrasts(self, groups, contrasts="pairs", batch=None, batch_models=None, n_randomizations: int = 150,
                  return_posteriors: bool = False, expectation=0, seed: int = 1, n_cores: int = 1,
                  chunked_draws: bool = False) -> dict:
        """``{"<A> vs <B>": result}``, each result what ``scde_expression_difference`` returns for that contrast (with
        the same n_cores and chunked_draws)."""
        if not self._ds:
            _stop("the session is closed")
        draw_chunks = _draw_chunks(chunked_draws, n_cores, None)
        gcodes, glev = _named_factor(groups, self.models.index)
        plan = expand_contrasts(glev, contrasts)
        code_of = {lev: i for i, lev in enumerate(glev)}
        sides, side_id, pairs = [], {}, []
        for label, la, lb, _na, _nb in plan:
            ids = []
            for lv in (la, lb):
                key = tuple(sorted(code_of[v] for v in lv))
                if key not in side_id:
                    cells = np.nonzero(np.isin(gcodes, key))[0].astype(np.int32)
                    if len(cells) == 0:
                        _stop(f"no cells in {_side_label(lv)} (contrast {label})")
                    side_id[key] = len(sides)
                    sides.append(cells)
                ids.append(side_id[key])
            pairs += ids
        correct_batch, bcodes, blev = False, None, []
        if batch is not None:
            bcodes, blev = _named_factor(batch, self.models.index)
            correct_batch = len(blev) > 1
        bmm, blt, bsq = _batch_model_matrix(self.models, batch_models) if correct_batch else (None, 0, 0)
        if correct_batch:  # the warning of R/functions.R:336-349, per contrast
            for label, la, lb, _na, _nb in plan:
                ia, ib = (sides[side_id[tuple(sorted(code_of[v] for v in lv))]] for lv in (la, lb))
                tab = np.array([np.bincount(bcodes[i][bcodes[i] >= 0], minlength=len(blev)) for i in (ia, ib)])
                pval = fisher_test_p_value(tab)
                if pval < 1e-3:
                    sys.stdout.write(f"WARNING: strong interaction between groups and batches in {label}! "
                                     "Correction may be ineffective:\n")
                    sys.stdout.write(f"Fisher's Exact Test for Count Data: p-value = {pval:.4g}\n")
        diffv, zi, adiffv, zia = _zero_indices(self._x, expectation, self.G)
        nc, ng, G, K = len(plan), len(sides), self.G, self.K
        off = np.zeros(ng + 1, dtype=np.int32)
        off[1:] = np.cumsum([len(s) for s in sides])
        cells = np.concatenate(sides).astype(np.int32)
        pr = np.asarray(pairs, dtype=np.int32)
        a = _lib.ContrastArgs()
        a.n_groups, a.group_offsets, a.group_cells = ng, p_i32(off), p_i32(cells)
        a.n_contrasts, a.pairs = nc, p_i32(pr)
        a.n_boot, a.seed = int(n_randomizations), int(seed)
        a.draw_chunks = draw_chunks
        zi, zia = i32(zi), i32(zia)
        a.zero_index, a.n_zero, a.zero_index_adjusted = p_i32(zi), len(zi), p_i32(zia)
        bc = i32(bcodes) if correct_batch else None
        a.batch, a.n_batch_levels = p_i32(bc), len(blev) if correct_batch else 0
        if bmm is not None:
            a.batch_models, a.batch_local_theta, a.batch_square_logit_conc = p_f64(bmm), blt, bsq
        o = _lib.ContrastOut()
        r = {"idx": np.empty((nc, 3, G), np.int32), "z": np.empty((nc, G)), "cz": np.empty((nc, G))}
        o.idx, o.z, o.cz = p_i32(r["idx"]), p_f64(r["z"]), p_f64(r["cz"])
        if correct_batch:
            for k in ("batch", "adjusted"):
                r[k + "_idx"], r[k + "_z"], r[k + "_cz"] = np.empty((nc, 3, G), np.int32), np.empty((nc, G)), np.empty((nc, G))
                setattr(o, k + "_idx", p_i32(r[k + "_idx"]))
                setattr(o, k + "_z", p_f64(r[k + "_z"]))
                setattr(o, k + "_cz", p_f64(r[k + "_cz"]))
        if return_posteriors:
            r["difference_posterior"] = np.empty((nc, 2 * K - 1, G))
            r["jp"] = np.empty((ng, K, G))
            o.difference_posterior, o.joint_posteriors = p_f64(r["difference_posterior"]), p_f64(r["jp"])
            if correct_batch:
                r["adjusted_difference_posterior"] = np.empty((nc, 4 * K - 3, G))
                o.adjusted_difference_posterior = p_f64(r["adjusted_difference_posterior"])
        st = _lib.Stats()
        check(lib().scde_b200_dataset_contrasts(self.ctx.handle, self._ds, C.byref(a), C.byref(o), C.byref(st)))
        self.last_stats = st.as_dict()
        out = {}
        for c, (label, _la, _lb, na, nb) in enumerate(plan):
            rc = {k: (v[c].T if v.ndim == 3 else v[c]) for k, v in r.items() if k != "jp"}
            if return_posteriors:
                rc["joint_posteriors"] = [r["jp"][pairs[2 * c]].T, r["jp"][pairs[2 * c + 1]].T]
            out[label] = _difference_result(rc, self.genes, diffv, adiffv, self._kcols, (na, nb), correct_batch,
                                            return_posteriors, self.last_stats)
        return out

    def close(self):
        if getattr(self, "_ds", None):
            lib().scde_b200_dataset_free(self.ctx.handle, self._ds)
            self._ds = C.c_void_p()

    def __enter__(self):
        return self

    def __exit__(self, *exc):
        self.close()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


def scde_expression_difference_contrasts(models: pd.DataFrame, counts, prior, groups, contrasts="pairs", batch=None,
                                         batch_models=None, n_randomizations: int = 150, return_posteriors: bool = False,
                                         expectation=0, seed: int = 1, context=None, n_cores: int = 1,
                                         chunked_draws: bool = False) -> dict:
    """scde.expression.difference for every contrast of `groups` (``"pairs"``, ``"rest"`` or a list of pairs; see
    ``expand_contrasts``) in one device session: ``{"<A> vs <B>": result}``."""
    with DifferenceSession(models, counts, prior, context=context) as s:
        return s.contrasts(groups, contrasts=contrasts, batch=batch, batch_models=batch_models,
                           n_randomizations=n_randomizations, return_posteriors=return_posteriors,
                           expectation=expectation, seed=seed, n_cores=n_cores, chunked_draws=chunked_draws)
