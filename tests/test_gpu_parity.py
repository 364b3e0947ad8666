"""GPU parity tests: the CUDA path, called through the C ABI, against the CPU oracle on identical inputs
(same bootstrap draws).  Tolerances (BASELINE.json north star): bootstrap indices bit-exact; log-posteriors within
1e-6 relative; lb/ub within one grid step (asserted exactly here and reported if not); mle index exact; Z within 1e-6."""
import ctypes as C

import numpy as np
import pandas as pd
import pytest

import helpers
from oracle import oracle as O
from scde_b200 import _lib, api, synth

pytestmark = pytest.mark.gpu

LOGP_RTOL = 1e-6


def _logp_close(a, b, rtol=LOGP_RTOL, floor=1e-290):
    """|log a - log b| <= rtol * |log b| wherever both are above the underflow floor; absolute 1e-300 elsewhere."""
    a, b = np.asarray(a), np.asarray(b)
    big = (a > floor) & (b > floor)
    la, lb = np.log(a[big]), np.log(b[big])
    ok_big = np.all(np.abs(la - lb) <= rtol * np.maximum(np.abs(lb), 1.0))
    ok_small = np.all(np.abs(a[~big] - b[~big]) <= 1e-280)
    worst = float(np.max(np.abs(la - lb) / np.maximum(np.abs(lb), 1.0))) if big.any() else 0.0
    return bool(ok_big and ok_small), worst


def _z_close(got, want):
    """Z within 1e-6, except below about -6: there the reference's own formula takes the upper tail of gs = 1 - 4e-13
    (R/functions.R:3528), so one ulp of gs (1.1e-16; long double vs double-double accumulation) is 4e-5 in Z."""
    got, want = np.asarray(got, dtype=np.float64), np.asarray(want, dtype=np.float64)
    tol = np.where(want < -6.0, 2e-4, 1e-6 * np.maximum(1.0, np.abs(want)) + 1e-9)
    bad = np.abs(got - want) > tol
    assert not bad.any(), f"Z mismatch: max |dZ| = {np.max(np.abs(got - want)):.3e} at {np.argmax(np.abs(got - want))}"


def _rows_close(got, want):
    """Table rows: 1e-9 where exp() of the value is a normal double; below -700 the reference's own exp(nb - max) is a
    denormal with one to a few significant bits, so a 1e-13 change of its argument can flip the last bit (log 2 at
    worst) or, at the very end of the range (< -735), flip between the smallest denormal and zero, i.e. between a
    finite value and the "log 0" clamp.  The clamp value itself must be exact."""
    sent_w, sent_g = want < -1e300, got < -1e300
    both = sent_w & sent_g
    assert np.array_equal(want[both], got[both])
    flip = sent_w ^ sent_g
    if flip.any():
        finite_side = np.where(sent_w, got, want)[flip]
        assert np.all(finite_side < -735.0), "clamp position differs outside the denormal underflow edge"
    ok = ~sent_w & ~sent_g
    norm = ok & (want > -700.0)
    np.testing.assert_allclose(got[norm], want[norm], rtol=1e-9, atol=1e-9)
    den = ok & ~norm
    if den.any():
        assert np.max(np.abs(got[den] - want[den])) <= 0.7


def _small_problem(G=97, Cn=23, seed=5, batch=False):
    w = synth.make_workload(3, n_genes=G, n_cells=Cn, batch=batch, seed=seed)
    return w


def _oracle_inputs(w):
    mm, lt, sq = O.pack_models(w.models)
    mag = O.marginals_from_prior_x(w.prior["x"].to_numpy())
    return mm, lt, sq, mag


# ------------------------------------------------------------------------------------------------
def test_cell_table_matches_oracle(ctx):
    ifm = helpers.o_ifm()
    cd, _, prior, _ = helpers.es_mef_inputs("tests")
    mm, lt, sq = O.pack_models(ifm)
    mag = O.marginals_from_prior_x(prior["x"].to_numpy())
    for cell in (0, 7, 39):
        uc = np.unique(cd.to_numpy()[:, cell]).astype(np.int32)
        want, wmodes = O.cell_table(mm[cell], uc, mag, ncells_for_clamp=20)
        got = np.empty((len(uc), len(mag)))
        gmodes = np.empty(len(uc), np.int32)
        _lib.check(_lib.lib().scde_b200_cell_table(ctx.handle, _lib.p_f64(_lib.f64(mm[cell])), _lib.p_i32(uc), len(uc),
                                                   _lib.p_f64(_lib.f64(mag)), len(mag), 0, 0, 20, _lib.p_f64(got),
                                                   _lib.p_i32(gmodes)))
        _rows_close(got, want.T)
        assert np.array_equal(gmodes, wmodes)


def test_cell_table_local_theta(ctx):
    knn = helpers.knn_models()
    mm, lt, sq = O.pack_models(knn)
    assert lt == 1 and sq == 1
    mag = O.marginals_from_prior_x(np.linspace(0, 4.8, 401))
    uc = np.array([0, 1, 2, 3, 7, 19, 150, 2048, 99999], dtype=np.int32)
    for cell in (0, 31, 63):
        want, wmodes = O.cell_table(mm[cell], uc, mag, localtheta=1, sqlogit=1, ncells_for_clamp=64)
        got = np.empty((len(uc), len(mag)))
        gmodes = np.empty(len(uc), np.int32)
        _lib.check(_lib.lib().scde_b200_cell_table(ctx.handle, _lib.p_f64(_lib.f64(mm[cell])), _lib.p_i32(uc), len(uc),
                                                   _lib.p_f64(_lib.f64(mag)), len(mag), 1, 1, 64, _lib.p_f64(got),
                                                   _lib.p_i32(gmodes)))
        _rows_close(got, want.T)
        assert np.array_equal(gmodes, wmodes)


@pytest.mark.parametrize("kernel", [1, 2, 3])  # generic FP64, tiled FP64 (DMMA), tcgen05 int8 fixed point
@pytest.mark.parametrize("G,Cn,B", [(97, 23, 100), (5, 1, 7), (33, 40, 150), (1, 9, 100)])
def test_posteriors_match_oracle(ctx, kernel, G, Cn, B):
    w = _small_problem(G, Cn)
    mm, lt, sq, mag = _oracle_inputs(w)
    flat, off, uci = O.unique_counts(w.counts)
    bi = O.boot_indices(1, Cn, B)
    want = O.log_boot_posterior(mm, flat, off, uci, mag, B, boot_idx=bi)["jp"]
    ctx.set_contract_kernel(kernel)
    try:
        got = api.scde_posteriors(w.models, w.counts, w.prior, n_randomizations=B, context=ctx)
    finally:
        ctx.set_contract_kernel(0)
    ok, worst = _logp_close(got.to_numpy(), want)
    assert ok, f"log-posterior mismatch, worst relative {worst:.3e}"
    np.testing.assert_allclose(got.to_numpy().sum(axis=1), 1.0, rtol=1e-12)


def test_posteriors_variants(ctx):
    w = _small_problem(41, 12)
    mm, lt, sq, mag = _oracle_inputs(w)
    flat, off, uci = O.unique_counts(w.counts)
    # no bootstrap
    want = O.log_boot_posterior(mm, flat, off, uci, mag, 0)["jp"]
    got = api.scde_posteriors(w.models, w.counts, w.prior, n_randomizations=0, context=ctx)
    assert _logp_close(got.to_numpy(), want)[0]
    # ensemble
    want = O.log_boot_posterior(mm, flat, off, uci, mag, 10, ensemble=1)["jp"]
    got = api.scde_posteriors(w.models, w.counts, w.prior, n_randomizations=10, ensemble_posterior=True, context=ctx)
    np.testing.assert_allclose(got.to_numpy(), want, rtol=1e-9, atol=1e-300)
    # modes + individual posteriors
    ow = O.log_boot_posterior(mm, flat, off, uci, mag, 20, returnpost=3)
    gw = api.scde_posteriors(w.models, w.counts, w.prior, n_randomizations=20, return_individual_posteriors=True,
                             return_individual_posterior_modes=True, context=ctx)
    assert _logp_close(gw["jp"].to_numpy(), ow["jp"])[0]
    np.testing.assert_array_equal(gw["modes"].to_numpy(), ow["modes"])
    for i, cell in enumerate(w.models.index):
        _rows_close(gw["post"][cell].to_numpy(), ow["post"][i])


def test_batch_posteriors_match_oracle(ctx):
    w = _small_problem(53, 31, batch=True)
    mm, lt, sq, mag = _oracle_inputs(w)
    flat, off, uci = O.unique_counts(w.counts)
    bcodes = np.asarray(w.batch.codes)
    pools = [np.nonzero(bcodes == l)[0].astype(np.int32) for l in range(2)]
    comp = np.array([5, 0], dtype=np.int32)  # a zero-count composition level
    want = O.log_boot_batch_posterior(mm, flat, off, uci, mag, pools, comp, 40, seed=1)["jp"]
    got = api.scde_posteriors(w.models, w.counts, w.prior, n_randomizations=40, batch=w.batch,
                              composition={"batch1": 5, "batch2": 0}, context=ctx)
    assert _logp_close(got.to_numpy(), want)[0]
    comp = np.bincount(bcodes[:15], minlength=2).astype(np.int32)
    want = O.log_boot_batch_posterior(mm, flat, off, uci, mag, pools, comp, 100, seed=1)["jp"]
    got = api.scde_posteriors(w.models, w.counts, w.prior, n_randomizations=100, batch=w.batch, composition=comp,
                              context=ctx)
    assert _logp_close(got.to_numpy(), want)[0]


def test_mat_slide_mult_bit_exact(ctx):
    rng = np.random.default_rng(3)
    for G, n in [(7, 5), (64, 401), (3, 801), (1, 1)]:
        a, b = rng.random((G, n)), rng.random((G, n)) * 1e-3
        want = O.mat_slide_mult(a, b)
        got = api.mat_slide_mult(a, b, context=ctx)
        assert np.array_equal(got, want)  # separately rounded multiply/add in ascending j: bit-identical
        ref = np.stack([np.correlate(a[g], b[g], "full") for g in range(G)])
        np.testing.assert_allclose(got, ref, rtol=1e-12)


def test_legacy_jpmat_log_boot(ctx):
    rng = np.random.default_rng(11)
    matl = [np.log(rng.dirichlet(np.ones(37), size=19)) for _ in range(6)]
    bi = O.boot_indices(3, 6, 25)
    want = O.jpmat_log_boot(matl, 25, seed=3)
    got = api.jpmat_log_boot(matl, 25, 3, context=ctx)
    np.testing.assert_allclose(got, want, rtol=1e-10)
    got2 = api.jpmat_log_boot(matl, 25, 3, boot_idx=bi, context=ctx)
    assert np.array_equal(got, got2)
    matll = [matl[:2], matl[2:]]
    want = O.jpmat_log_batch_boot(matll, [3, 2], 25, seed=4)
    got = api.jpmat_log_batch_boot(matll, [3, 2], 25, 4, context=ctx)
    np.testing.assert_allclose(got, want, rtol=1e-10)


def _compare_summaries(got: pd.DataFrame, want: np.ndarray, widx, gidx, what):
    assert np.array_equal(gidx[:, 1], widx[:, 1]), f"{what}: mle grid index differs"
    assert np.max(np.abs(gidx[:, [0, 2]] - widx[:, [0, 2]])) <= 1, f"{what}: bound differs by more than one grid step"
    assert np.array_equal(gidx, widx), f"{what}: bounds differ (within one step)"
    _z_close(got["Z"].to_numpy(), want[:, 4])
    _z_close(got["cZ"].to_numpy(), want[:, 5])
    np.testing.assert_allclose(got[["lb", "mle", "ub", "ce"]].to_numpy(), want[:, :4], rtol=1e-12, atol=1e-300)


def test_expression_difference_small(ctx):
    w = _small_problem(211, 30)
    codes = np.asarray(w.groups.codes)
    want = O.expression_difference(w.models, w.counts, w.prior["x"].to_numpy(), w.prior["y"].to_numpy(),
                                   (np.nonzero(codes == 0)[0], np.nonzero(codes == 1)[0]), nboot=100, seed=1)
    job_res = api.scde_expression_difference(w.models, w.counts, w.prior, groups=w.groups, n_randomizations=100,
                                             return_posteriors=True, context=ctx)
    got = job_res["results"]
    ok, worst = _logp_close(job_res["difference.posterior"].to_numpy(), want["difference.posterior"])
    assert ok, worst
    for i, lev in enumerate(["g1", "g2"]):
        assert _logp_close(job_res["joint.posteriors"][lev].to_numpy(), want["joint.posteriors"][i])[0]
    diffv = api.fold_change_grid(w.prior["x"].to_numpy())
    gidx = np.stack([np.searchsorted(diffv, got[c].to_numpy() * np.log10(2.0) - 1e-9) for c in ("lb", "mle", "ub")], 1)
    _compare_summaries(got, want["results"], want["idx"], gidx, "results")


def test_expression_difference_batch_small(ctx):
    w = _small_problem(101, 26, batch=True)
    codes = np.asarray(w.groups.codes)
    bcodes = np.asarray(w.batch.codes)
    ex = 0.5
    want = O.expression_difference(w.models, w.counts, w.prior["x"].to_numpy(), w.prior["y"].to_numpy(),
                                   (np.nonzero(codes == 0)[0], np.nonzero(codes == 1)[0]), nboot=60, seed=1,
                                   batch_codes=bcodes, expectation=ex)
    got = api.scde_expression_difference(w.models, w.counts, w.prior, groups=w.groups, batch=w.batch,
                                         n_randomizations=60, return_posteriors=True, expectation=ex, context=ctx)
    assert _logp_close(got["batch.adjusted.difference.posterior"].to_numpy(),
                       want["batch.adjusted.difference.posterior"])[0]
    for key in ("results", "batch.effect", "batch.adjusted"):
        _z_close(got[key]["Z"].to_numpy(), want[key][:, 4])
        np.testing.assert_allclose(got[key][["lb", "mle", "ub", "ce"]].to_numpy(), want[key][:, :4], rtol=1e-12,
                                   atol=1e-300)
        _z_close(got[key]["cZ"].to_numpy(), want[key][:, 5])


def test_expression_magnitude(ctx):
    cd, ifm, prior, groups = helpers.es_mef_inputs("tests")
    sub = cd.iloc[:500]
    got = api.scde_expression_magnitude(ifm, sub)
    with np.errstate(divide="ignore"):
        want = O.expression_magnitude(sub.to_numpy(), ifm["corr.b"].to_numpy(), ifm["corr.a"].to_numpy())
    assert np.array_equal(np.isneginf(got.to_numpy()), np.isneginf(want))
    fin = np.isfinite(want)
    np.testing.assert_allclose(got.to_numpy()[fin], want[fin], rtol=1e-14)


def test_es_mef_small_subset_full_path(ctx):
    """cfg1 (bundled data): a 1500-gene slice through the whole path against the oracle; the two FP64 kernels agree to
    rounding, the default (tcgen05 fixed-point) kernel agrees with them within the 1e-6 contract."""
    cd, ifm, prior, groups = helpers.es_mef_inputs("tests")
    sub = cd.iloc[2000:3500]
    codes = np.asarray(groups.codes)
    want = O.expression_difference(ifm, sub.to_numpy(), prior["x"].to_numpy(), prior["y"].to_numpy(),
                                   (np.nonzero(codes == 0)[0], np.nonzero(codes == 1)[0]), nboot=100, seed=1)
    got = api.scde_expression_difference(ifm, sub, prior, groups=groups, n_randomizations=100, context=ctx)
    _z_close(got["Z"].to_numpy(), want["results"][:, 4])
    np.testing.assert_allclose(got[["lb", "mle", "ub", "ce"]].to_numpy(), want["results"][:, :4], rtol=1e-12, atol=1e-300)
    by_kernel = {}
    for kernel in (1, 2):
        ctx.set_contract_kernel(kernel)
        try:
            by_kernel[kernel] = api.scde_expression_difference(ifm, sub, prior, groups=groups, n_randomizations=100,
                                                               context=ctx)
        finally:
            ctx.set_contract_kernel(0)
    np.testing.assert_allclose(by_kernel[1]["Z"].to_numpy(), by_kernel[2]["Z"].to_numpy(), rtol=1e-9, atol=1e-12)
    _z_close(got["Z"].to_numpy(), by_kernel[2]["Z"].to_numpy())
    assert np.array_equal(got[["lb", "mle", "ub"]].to_numpy(), by_kernel[2][["lb", "mle", "ub"]].to_numpy())


def test_error_paths(ctx):
    w = _small_problem(10, 6)
    with pytest.raises(ValueError):
        api.scde_expression_difference(w.models, w.counts[:, :3], w.prior, groups=w.groups, context=ctx)
    bad = w.counts.copy()
    bad[0, 0] = -4
    with pytest.raises(_lib.ScdeB200Error):
        api.scde_expression_difference(w.models, bad, w.prior, groups=w.groups, n_randomizations=5, context=ctx)
    with pytest.raises(ValueError):
        api.scde_expression_difference(w.models, w.counts, w.prior,
                                       groups=pd.Categorical(["a", "b", "c", "a", "b", "c"]), context=ctx)


def test_full_size_properties(ctx):
    """cfg3-sized shapes are too slow for the oracle; check size-independent properties instead: rows of the joint
    posterior sum to one, swapping the groups mirrors the summary, and an oracle spot-check on a gene subset."""
    w = synth.make_workload(3, n_genes=3000, n_cells=600)
    res = api.scde_expression_difference(w.models, w.counts, w.prior, groups=w.groups, n_randomizations=100,
                                         return_posteriors=True, context=ctx)
    for lev in ("g1", "g2"):
        np.testing.assert_allclose(res["joint.posteriors"][lev].to_numpy().sum(axis=1), 1.0, rtol=1e-11)
    np.testing.assert_allclose(res["difference.posterior"].to_numpy().sum(axis=1), 1.0, rtol=1e-11)
    swapped = pd.Categorical(np.where(np.asarray(w.groups.codes) == 0, "g2", "g1"), categories=["g1", "g2"])
    # same cells per level, levels exchanged -> the ratio posterior is mirrored (draws are per level size: equal halves)
    res2 = api.scde_expression_difference(w.models, w.counts, w.prior, groups=swapped, n_randomizations=100,
                                          return_posteriors=True, context=ctx)
    a = res["difference.posterior"].to_numpy()
    b = res2["difference.posterior"].to_numpy()[:, ::-1]
    np.testing.assert_allclose(a, b, rtol=1e-9, atol=1e-300)
    # Z is only approximately antisymmetric: the mirrored tail mass is 1 - gs - zv, which rounds differently
    np.testing.assert_allclose(res["results"]["Z"].to_numpy(), -res2["results"]["Z"].to_numpy(), rtol=1e-4, atol=1e-4)
    # oracle spot-check on 24 genes with the same draws
    sel = np.arange(0, 3000, 125)
    codes = np.asarray(w.groups.codes)
    want = O.expression_difference(w.models, w.counts[sel], w.prior["x"].to_numpy(), w.prior["y"].to_numpy(),
                                   (np.nonzero(codes == 0)[0], np.nonzero(codes == 1)[0]), nboot=100, seed=1)
    ok, worst = _logp_close(a[sel], want["difference.posterior"])
    assert ok, worst
    # cZ is global over genes, so compare Z only
    _z_close(res["results"]["Z"].to_numpy()[sel], want["results"][:, 4])


def test_es_mef_small_all_genes_against_committed_golden(ctx):
    """cfg1 on the real data, every gene: the CUDA path against the oracle output committed in tests/golden (vignette
    variant: G = 12142, max.quantile = 0.999, Seed = 1, 100 randomizations)."""
    import os
    d = np.load(os.path.join(helpers.GOLD, "es_mef_vignette_oracle.npz"))
    cd, ifm, prior, groups = helpers.es_mef_inputs("vignette")
    assert [str(g) for g in d["genes"]] == list(cd.index)
    got = api.scde_expression_difference(ifm, cd, prior, groups=groups, n_randomizations=100, context=ctx)
    want = d["results"]
    diffv = api.fold_change_grid(prior["x"].to_numpy())
    step = (diffv[1] - diffv[0]) / np.log10(2.0)
    dq = got[["lb", "mle", "ub"]].to_numpy() - want[:, :3]
    n_off = int(np.sum(np.abs(dq) > 1e-9))
    assert np.max(np.abs(dq)) <= step * 1.0001, "a bound or mle moved by more than one grid step"
    assert n_off == 0, f"{n_off} of {dq.size} lb/mle/ub grid indices differ from the oracle (each by one step)"
    _z_close(got["Z"].to_numpy(), want[:, 4])
    _z_close(got["cZ"].to_numpy(), want[:, 5])
    top = list(got.sort_values("Z", ascending=False).index[:6])
    assert len(set(top) & {"Dppa5a", "Pou5f1", "Gm13242", "Tdh", "Ift46", "4930509G22Rik"}) >= 5  # vignette rows


def test_knn_models_local_theta_full_path(ctx):
    """12-column models (local theta fit + conc.a2, data/knn.rda) through scde.posteriors with per-cell modes -- the
    pagoda.varnorm call shape (R/functions.R:1425)."""
    knn = helpers.knn_models().iloc[:12]
    rng = np.random.default_rng(8)
    counts = np.asfortranarray(rng.negative_binomial(0.6, 0.02, size=(60, 12)).astype(np.int32))
    counts[rng.random(counts.shape) < 0.4] = 0
    prior = synth.make_prior(60)
    mm, lt, sq = O.pack_models(knn)
    mag = O.marginals_from_prior_x(prior["x"].to_numpy())
    flat, off, uci = O.unique_counts(counts)
    want = O.log_boot_posterior(mm, flat, off, uci, mag, 30, seed=1, returnpost=1, localtheta=lt, sqlogit=sq)
    got = api.scde_posteriors(knn, counts, prior, n_randomizations=30, return_individual_posterior_modes=True, context=ctx)
    ok, worst = _logp_close(got["jp"].to_numpy(), want["jp"])
    assert ok, worst
    np.testing.assert_array_equal(got["modes"].to_numpy(), want["modes"])


def test_na_group_cells_and_per_gene_expectation(ctx):
    w = _small_problem(40, 18)
    codes = np.asarray(w.groups.codes).copy()
    codes[[2, 11]] = -1  # NA: in neither group
    groups = pd.Categorical.from_codes(codes, categories=["g1", "g2"])
    ex = np.linspace(-1.5, 1.5, 40)
    want = O.expression_difference(w.models, w.counts, w.prior["x"].to_numpy(), w.prior["y"].to_numpy(),
                                   (np.nonzero(codes == 0)[0], np.nonzero(codes == 1)[0]), nboot=50, seed=1, expectation=ex)
    got = api.scde_expression_difference(w.models, w.counts, w.prior, groups=groups, n_randomizations=50, expectation=ex,
                                         context=ctx)
    _z_close(got["Z"].to_numpy(), want["results"][:, 4])
    np.testing.assert_allclose(got[["lb", "mle", "ub", "ce"]].to_numpy(), want["results"][:, :4], rtol=1e-12, atol=1e-300)


def test_zero_base_equals_dense_form(ctx):
    """The zero-base contraction (visit only non-zero-count cells) against the dense form on the same device."""
    w = synth.make_workload(3, n_genes=300, n_cells=120, seed=4)
    ctx.set_contract_kernel(2)  # both forms on the FP64 kernel: they differ by rounding only
    try:
        a = api.scde_expression_difference(w.models, w.counts, w.prior, groups=w.groups, n_randomizations=100,
                                           return_posteriors=True, context=ctx)
        keep = ctx.set_options(zero_base=0)
        try:
            b = api.scde_expression_difference(w.models, w.counts, w.prior, groups=w.groups, n_randomizations=100,
                                               return_posteriors=True, context=ctx)
        finally:
            ctx.restore_options(keep)
    finally:
        ctx.set_contract_kernel(0)
    assert a["stats"]["contract_cells"] < 0.8 * b["stats"]["contract_cells"]
    for lev in ("g1", "g2"):
        ok, worst = _logp_close(a["joint.posteriors"][lev].to_numpy(), b["joint.posteriors"][lev].to_numpy(), rtol=1e-9)
        assert ok, worst
    assert np.array_equal(a["results"][["lb", "mle", "ub"]].to_numpy(), b["results"][["lb", "mle", "ub"]].to_numpy())


def test_batch_config5_shape_against_oracle_subset(ctx):
    w = synth.make_workload(5, n_genes=400, n_cells=300)
    codes = np.asarray(w.groups.codes)
    bcodes = np.asarray(w.batch.codes)
    got = api.scde_expression_difference(w.models, w.counts, w.prior, groups=w.groups, batch=w.batch, n_randomizations=100,
                                         context=ctx)
    sel = np.arange(0, 400, 25)
    want = O.expression_difference(w.models, w.counts[sel], w.prior["x"].to_numpy(), w.prior["y"].to_numpy(),
                                   (np.nonzero(codes == 0)[0], np.nonzero(codes == 1)[0]), nboot=100, seed=1,
                                   batch_codes=bcodes)
    for key in ("results", "batch.effect", "batch.adjusted"):
        _z_close(got[key]["Z"].to_numpy()[sel], want[key][:, 4])
        np.testing.assert_allclose(got[key][["lb", "mle", "ub"]].to_numpy()[sel], want[key][:, :3], rtol=1e-12, atol=1e-300)


def test_single_gene_test_tdh(ctx):
    """scde.test.gene.expression.difference("Tdh", ...) numeric core: G = 1, 1000 randomizations, individual posteriors
    (tests/tests.R:46, vignettes/diffexp.md:139: lb 5.73 mle 8.04 ub 10.30 Z 7.15 with another libc's rand())."""
    cd, ifm, prior, groups = helpers.es_mef_inputs("vignette")
    got = api.scde_test_gene_expression_difference("Tdh", ifm, cd, prior, groups=groups, return_details=True, context=ctx)
    codes = np.asarray(groups.codes)
    want = O.expression_difference(ifm, cd.loc[["Tdh"]].to_numpy(), prior["x"].to_numpy(), prior["y"].to_numpy(),
                                   (np.nonzero(codes == 0)[0], np.nonzero(codes == 1)[0]), nboot=1000, seed=1)
    r = got["results"]
    np.testing.assert_allclose(r[["lb", "mle", "ub", "ce"]].to_numpy(), want["results"][:, :4], rtol=1e-12)
    _z_close(r["Z"].to_numpy(), want["results"][:, 4])
    assert abs(r["Z"].iloc[0] - r["cZ"].iloc[0]) < 1e-12  # one gene: BH leaves Z unchanged
    ok, worst = _logp_close(got["difference.posterior"].to_numpy(), want["difference.posterior"])
    assert ok, worst
    step = 0.0397793
    assert abs(r["lb"].iloc[0] - 5.728235) <= 5 * step and abs(r["ub"].iloc[0] - 10.30287) <= 5 * step
    assert abs(r["Z"].iloc[0] - 7.151425) < 0.05
    assert set(got["posteriors"]) == {"ESC", "MEF"} and len(got["posteriors"]["ESC"]["post"]) == 20


@pytest.mark.parametrize("length_out", [200, 500])
def test_other_grid_sizes(ctx, length_out):
    """K = 201 (tiled kernel, half-empty tiles) and K = 501 (> 416: generic contraction kernel, general table stride)."""
    w = _small_problem(45, 14)
    prior = synth.make_prior(45, length_out=length_out)
    codes = np.asarray(w.groups.codes)
    want = O.expression_difference(w.models, w.counts, prior["x"].to_numpy(), prior["y"].to_numpy(),
                                   (np.nonzero(codes == 0)[0], np.nonzero(codes == 1)[0]), nboot=30, seed=1)
    got = api.scde_expression_difference(w.models, w.counts, prior, groups=w.groups, n_randomizations=30,
                                         return_posteriors=True, context=ctx)
    ok, worst = _logp_close(got["difference.posterior"].to_numpy(), want["difference.posterior"])
    assert ok, worst
    _z_close(got["results"]["Z"].to_numpy(), want["results"][:, 4])
    np.testing.assert_allclose(got["results"][["lb", "mle", "ub"]].to_numpy(), want["results"][:, :3], rtol=1e-12, atol=1e-300)


def test_all_zero_and_constant_genes(ctx):
    """Genes whose counts are all zero (empty entry list: T is the base sum alone) and genes with one non-zero cell."""
    w = _small_problem(30, 16)
    counts = w.counts.copy()
    counts[0, :] = 0
    counts[1, :] = 0
    counts[1, 5] = 7
    counts[2, :] = 3
    codes = np.asarray(w.groups.codes)
    want = O.expression_difference(w.models, counts, w.prior["x"].to_numpy(), w.prior["y"].to_numpy(),
                                   (np.nonzero(codes == 0)[0], np.nonzero(codes == 1)[0]), nboot=100, seed=1)
    got = api.scde_expression_difference(w.models, counts, w.prior, groups=w.groups, n_randomizations=100,
                                         return_posteriors=True, context=ctx)
    for i, lev in enumerate(["g1", "g2"]):
        ok, worst = _logp_close(got["joint.posteriors"][lev].to_numpy(), want["joint.posteriors"][i])
        assert ok, (lev, worst)
    _z_close(got["results"]["Z"].to_numpy(), want["results"][:, 4])


def test_single_randomization_and_single_cell_groups(ctx):
    w = _small_problem(12, 2)
    codes = np.asarray(w.groups.codes)
    want = O.expression_difference(w.models, w.counts, w.prior["x"].to_numpy(), w.prior["y"].to_numpy(),
                                   (np.nonzero(codes == 0)[0], np.nonzero(codes == 1)[0]), nboot=1, seed=1)
    got = api.scde_expression_difference(w.models, w.counts, w.prior, groups=w.groups, n_randomizations=1, context=ctx)
    _z_close(got["Z"].to_numpy(), want["results"][:, 4])
    np.testing.assert_allclose(got[["lb", "mle", "ub"]].to_numpy(), want["results"][:, :3], rtol=1e-12, atol=1e-300)


def _call_and_job(ctx, w, counts, **kw):
    """the one-shot C-ABI call (chunked upload overlapped with the table build) and the upload / run / download job"""
    mm, lt, sq = api.pack_models(w.models)
    x, y = w.prior["x"].to_numpy(), w.prior["y"].to_numpy()
    codes = np.asarray(w.groups.codes, dtype=np.int32)
    zi = api._zero_index(api.fold_change_grid(x), 0.0)
    one = api.expression_difference_call(ctx, counts, mm, x, y, codes, 100, 1, zero_index=zi, local_theta=lt, sqlogit=sq,
                                         joint_posteriors=True, **kw)
    job = api.DifferenceJob(ctx, counts, mm, x, y, codes, 100, 1, zero_index=zi, local_theta=lt, sqlogit=sq, **kw)
    try:
        job.run()
        two = job.download(joint_posteriors=True)
    finally:
        job.close()
    return one, two


def test_one_shot_call_pipelined_front_equals_job(ctx):
    """640 cells go up in seven chunks of 96; every chunk is deduplicated and its rows are built while the next ones are
    still in flight.  Row numbering, table and results must be those of the resident-counts path, bit for bit."""
    w = synth.make_workload(3, n_genes=150, n_cells=640, seed=21)
    one, two = _call_and_job(ctx, w, np.asarray(w.counts, dtype=np.int32, order="F"))
    assert one["stats"]["table_rows"] == two["stats"]["table_rows"]
    assert np.array_equal(one["idx"], two["idx"])
    assert np.array_equal(one["z"], two["z"])
    for i in range(2):
        assert np.array_equal(one["joint_posteriors"][i], two["joint_posteriors"][i])


def test_one_shot_call_gene_shard_and_row_estimate_fallback(ctx):
    """a gene shard of a wider matrix (strided upload), with the first chunk of cells all-zero: the row estimate made from
    that chunk is far too small, the kernels stop at the capacity and the library rebuilds index and table from the
    resident counts -- same results as the job path"""
    w = synth.make_workload(3, n_genes=200, n_cells=640, seed=22)
    counts = np.array(w.counts, dtype=np.int32, order="F")
    counts[:, :96] = 0
    counts[:, 96:] += np.arange(200, dtype=np.int32)[:, None] * 37  # hundreds of distinct counts per cell
    ctx = _lib.Context(0)  # a fresh workspace: no row buffers left over from a larger problem
    one, two = _call_and_job(ctx, w, counts, gene_range=(40, 190))
    assert one["stats"]["table_rows"] == two["stats"]["table_rows"] > 5000
    assert np.array_equal(one["idx"], two["idx"])
    assert np.array_equal(one["z"], two["z"])
    for i in range(2):
        assert np.array_equal(one["joint_posteriors"][i], two["joint_posteriors"][i])


def _assert_same(one, two):
    assert one["stats"]["table_rows"] == two["stats"]["table_rows"]
    assert np.array_equal(one["idx"], two["idx"])
    assert np.array_equal(one["z"], two["z"])
    for i in range(2):
        assert np.array_equal(one["joint_posteriors"][i], two["joint_posteriors"][i])


def test_one_shot_call_split_front_overflow_after_first_joint():
    """split front: the first group's cells hold a handful of distinct counts, so their rows fit the estimate and the first
    joint runs early; the second group's cells hold hundreds, the rest of the front hits the capacity, the table is
    rebuilt from the resident counts and the first joint is repeated on the new row ids -- same results as the job path"""
    w = synth.make_workload(3, n_genes=200, n_cells=640, seed=23)
    counts = np.array(w.counts, dtype=np.int32, order="F")
    counts[:, :320] = np.minimum(counts[:, :320], 2)
    counts[:, 320:] += np.arange(200, dtype=np.int32)[:, None] * 37
    ctx = _lib.Context(0)  # a fresh workspace: no row buffers left over from a larger problem
    one, two = _call_and_job(ctx, w, counts)
    assert one["stats"]["table_rows"] > 20000
    _assert_same(one, two)


def test_one_shot_call_group_layouts(ctx):
    """where the first group's cells lie decides whether the front is split: interleaved groups (no split), the first
    group in the trailing cells (no split), a short first group (split after a quarter), cells outside both groups"""
    w = synth.make_workload(3, n_genes=120, n_cells=640, seed=24)
    counts = np.asarray(w.counts, dtype=np.int32, order="F")
    base = np.asarray(w.groups.codes, dtype=np.int32)
    layouts = {
        "interleaved": (np.arange(640) % 2).astype(np.int32),
        "reversed": (1 - base).astype(np.int32),
        "short_first": np.where(np.arange(640) < 150, 0, 1).astype(np.int32),
        "with_na": np.where(np.arange(640) % 7 == 3, -1, base).astype(np.int32),
    }
    mm, lt, sq = api.pack_models(w.models)
    x, y = w.prior["x"].to_numpy(), w.prior["y"].to_numpy()
    zi = api._zero_index(api.fold_change_grid(x), 0.0)
    for name, codes in layouts.items():
        one = api.expression_difference_call(ctx, counts, mm, x, y, codes, 100, 1, zero_index=zi, local_theta=lt, sqlogit=sq,
                                             joint_posteriors=True)
        job = api.DifferenceJob(ctx, counts, mm, x, y, codes, 100, 1, zero_index=zi, local_theta=lt, sqlogit=sq)
        try:
            job.run()
            two = job.download(joint_posteriors=True)
        finally:
            job.close()
        _assert_same(one, two)


def test_one_shot_call_split_front_with_batch(ctx):
    """batch-corrected call through the split front: the two composition-sampled joints need every cell and run after the
    whole front; every array the call returns equals the job path's, bit for bit"""
    w = synth.make_workload(5, n_genes=100, n_cells=640, seed=25)
    counts = np.asarray(w.counts, dtype=np.int32, order="F")
    bcodes = np.asarray(w.batch.codes, dtype=np.int32)
    kw = dict(batch_codes=bcodes, n_batch_levels=int(bcodes.max()) + 1)
    one, two = _call_and_job(ctx, w, counts, **kw)
    n_cmp = 0
    for k, v in one.items():
        if isinstance(v, np.ndarray) and not k.endswith("cz"):  # cZ (BH over the call's genes) is an output of the one-shot call only
            assert np.array_equal(v, two[k]), k
            n_cmp += 1
    assert n_cmp >= 4


def test_dedup_bitmap_and_hash_cells_mixed(ctx):
    """cells whose counts all lie below 65536 are indexed by the bitmap kernels (eight cells per CTA), cells with a larger
    count by the hash kernels; both kinds side by side, a ragged last group of cells, against the oracle"""
    w = synth.make_workload(3, n_genes=120, n_cells=21, seed=31)
    counts = np.array(w.counts, dtype=np.int32, order="F")
    rng = np.random.default_rng(5)
    counts[:30, 3] = rng.integers(65536, 400000, size=30)   # cell 3 and cell 17 leave the bitmap range
    counts[5, 17] = 65536
    counts[:, 9] = 0                                         # a cell with the single distinct count 0
    # a few distinct counts beyond the bitmap stay with the bitmap kernels (overflow list, at most six per cell): one value
    # repeated in many genes, and four values up to the largest the count type holds, next to small counts
    counts[40:100, 12] = 70000
    counts[:4, 14] = [65536, 1_000_000, 65537, 2_000_000_000]
    counts[4:11, 15] = [65536, 65537, 65538, 65539, 65540, 65541, 65542]  # seven: one too many, the hash kernel again
    counts[7, 20] = 65535                                    # the last value the bitmap holds
    mm, lt, sq = api.pack_models(w.models)
    mag = api.marginals_from_prior(w.prior)
    flat, off, uci = O.unique_counts(counts)
    bi = O.boot_indices(1, counts.shape[1], 100)
    want = O.log_boot_posterior(mm, flat, off, uci, mag, 100, boot_idx=bi)["jp"]
    x, y = w.prior["x"].to_numpy(), w.prior["y"].to_numpy()
    codes = np.zeros(counts.shape[1], dtype=np.int32)
    codes[11:] = 1
    zi = api._zero_index(api.fold_change_grid(x), 0.0)
    # the fused call builds the index on the device from the raw counts (scde_posteriors takes the caller's ucl / uci)
    res = api.expression_difference_call(ctx, counts, mm, x, y, codes, 100, 1, zero_index=zi, local_theta=lt, sqlogit=sq,
                                         joint_posteriors=True)
    # the device gives every cell a zero-count row whether or not a gene has a zero there
    assert len(flat) <= res["stats"]["table_rows"] <= len(flat) + counts.shape[1]
    for lev in (0, 1):
        ii = np.nonzero(codes == lev)[0]
        fl, of, uc = O.unique_counts(counts[:, ii])
        wj = O.log_boot_posterior(np.asfortranarray(mm[ii]), fl, of, uc, mag, 100,
                                  boot_idx=O.boot_indices(1, len(ii), 100))["jp"]
        ok, worst = _logp_close(res["joint_posteriors"][lev], wj)
        assert ok, worst
    assert want.shape == (120, len(mag))


def _oracle_diff(w, nboot=100, batch_codes=None):
    codes = np.asarray(w.groups.codes)
    return O.expression_difference(w.models, w.counts, w.prior["x"].to_numpy(), w.prior["y"].to_numpy(),
                                   (np.nonzero(codes == 0)[0], np.nonzero(codes == 1)[0]), nboot=nboot, seed=1,
                                   batch_codes=batch_codes)


def test_gene_shard_against_oracle(ctx):
    """the shard path (gene_begin / gene_end of the one-shot call and of the job) against the ORACLE's rows of the same
    genes -- not against the library's own unsharded run: genes are independent, the draws are those of Seed = 1 whatever
    the range (n.cores = 1 semantics, SURVEY.md section 8(e))"""
    w = synth.make_workload(3, n_genes=230, n_cells=96, seed=31)
    want = _oracle_diff(w)
    mm, lt, sq = api.pack_models(w.models)
    x, y = w.prior["x"].to_numpy(), w.prior["y"].to_numpy()
    codes = np.asarray(w.groups.codes, dtype=np.int32)
    for g0, g1 in ((0, 77), (77, 154), (154, 230), (229, 230)):
        one = api.expression_difference_call(ctx, w.counts, mm, x, y, codes, 100, 1, local_theta=lt, sqlogit=sq,
                                             gene_range=(g0, g1), want_posteriors=True)
        assert np.array_equal(one["idx"], want["idx"][g0:g1])
        _z_close(one["z"], want["results"][g0:g1, 4])
        ok, worst = _logp_close(one["difference_posterior"], want["difference.posterior"][g0:g1])
        assert ok, worst
        job = api.DifferenceJob(ctx, w.counts, mm, x, y, codes, 100, 1, local_theta=lt, sqlogit=sq, gene_range=(g0, g1))
        try:
            job.run()
            two = job.download()
        finally:
            job.close()
        assert np.array_equal(two["idx"], one["idx"]) and np.array_equal(two["z"], one["z"])


def _multi_ctx(n):
    if _lib.lib().scde_b200_device_count() < n:
        pytest.skip(f"needs {n} CUDA devices")
    return _lib.Context(devices=list(range(n)))


@pytest.mark.parametrize("batch", [False, True])
def test_multi_device_call_equals_single_device(ctx, batch):
    """scde_b200_create_multi: the one-shot call shards the genes over two devices on two host threads and writes every
    shard's rows of the caller's buffers; bit-identical to the one-device call (the reference's n.cores > 1 would reseed
    per chunk, R/functions.R:613 -- the library keeps the n.cores = 1 draws), and within tolerance of the oracle."""
    mctx = _multi_ctx(2)
    w = synth.make_workload(5 if batch else 3, n_genes=301, n_cells=128, seed=41, batch=batch)
    mm, lt, sq = api.pack_models(w.models)
    x, y = w.prior["x"].to_numpy(), w.prior["y"].to_numpy()
    codes = np.asarray(w.groups.codes, dtype=np.int32)
    bc = np.asarray(w.batch.codes, dtype=np.int32) if batch else None
    kw = dict(batch_codes=bc, n_batch_levels=2 if batch else 0, local_theta=lt, sqlogit=sq, want_posteriors=True)
    if batch:
        kw["zero_index_adjusted"] = [2 * len(x) - 1]
    one = api.expression_difference_call(ctx, w.counts, mm, x, y, codes, 100, 1, **kw)
    two = api.expression_difference_call(mctx, w.counts, mm, x, y, codes, 100, 1, **kw)
    keys = ["idx", "z", "difference_posterior"] + (["adjusted_idx", "adjusted_z", "batch_idx", "batch_z",
                                                   "adjusted_difference_posterior"] if batch else [])
    for k in keys:
        assert np.array_equal(one[k], two[k]), k
    for i in range(2):
        assert np.array_equal(one["joint_posteriors"][i], two["joint_posteriors"][i])
    want = _oracle_diff(w, batch_codes=bc)
    assert np.array_equal(two["idx"], want["idx"])
    _z_close(two["z"], want["results"][:, 4])
    # a sub-range of the genes on the multi-device context, and fewer genes than devices
    sub = api.expression_difference_call(mctx, w.counts, mm, x, y, codes, 100, 1, gene_range=(100, 233), **kw)
    assert np.array_equal(sub["idx"], one["idx"][100:233]) and np.array_equal(sub["z"], one["z"][100:233])
    tiny = api.expression_difference_call(mctx, w.counts, mm, x, y, codes, 100, 1, gene_range=(300, 301), **kw)
    assert np.array_equal(tiny["z"], one["z"][300:301])
    mctx.close()


def test_second_device_runs_every_kernel(ctx):
    """function attributes (dynamic shared memory opt-in) are per device: a context on device 1 must be able to launch the
    tcgen05 and the FP64 contraction kernels after device 0 has (ADVICE r1: static attr_set)"""
    if _lib.lib().scde_b200_device_count() < 2:
        pytest.skip("needs 2 CUDA devices")
    w = synth.make_workload(3, n_genes=64, n_cells=40, seed=9)
    c1 = _lib.Context(1)
    for kernel in (0, 2, 1):
        res = []
        for c in (ctx, c1):
            c.set_contract_kernel(kernel)
            try:
                res.append(api.scde_posteriors(w.models, w.counts, w.prior, n_randomizations=20, context=c).to_numpy())
            finally:
                c.set_contract_kernel(0)
        assert np.array_equal(res[0], res[1])
    c1.close()


def test_cuda_path_against_reference_fixtures(ctx):
    """The CUDA path against outputs of THE REFERENCE'S OWN C++ (tests/golden/ref_fixtures_*.npz: src/jpmatLogBoot.cpp and
    src/matSlideMult.cpp compiled unmodified, tests/golden/make_ref_fixtures.py) -- no oracle in between.  Config 1's
    data incl. the vignette's six genes, a batch case, the 12-column knn models.  Log-posteriors 1e-6 relative, modes
    exact, matSlideMult bit-exact."""
    fx = helpers.ref_fixtures()
    sub, ifm, prior, groups, sel = helpers.ref_cfg1_inputs()
    codes = np.asarray(groups.codes)
    jps = []
    for lev in (0, 1):
        ii = np.nonzero(codes == lev)[0]
        r = api.scde_posteriors(ifm.iloc[ii], sub.iloc[:, ii], prior, n_randomizations=100,
                                return_individual_posterior_modes=True, context=ctx)
        ok, worst = _logp_close(r["jp"].to_numpy(), fx[f"cfg1_jp{lev}"])
        assert ok, worst
        assert np.array_equal(r["modes"].to_numpy(), fx[f"cfg1_modes{lev}"])
        jps.append(fx[f"cfg1_jp{lev}"])
    py = prior["y"].to_numpy()
    got = api.mat_slide_mult(jps[0] * py[None, :], jps[1] * py[None, :], context=ctx)
    assert np.array_equal(got, fx["cfg1_slide"])
    # the fused call on the same genes: joint posteriors of both groups against the reference's
    res = api.scde_expression_difference(ifm, sub, prior, groups=groups, n_randomizations=100, return_posteriors=True,
                                         context=ctx)
    for lev, name in enumerate(["ESC", "MEF"]):
        ok, worst = _logp_close(res["joint.posteriors"][name].to_numpy(), fx[f"cfg1_jp{lev}"])
        assert ok, worst
    w = helpers.ref_batch_inputs()
    res = api.scde_expression_difference(w.models, w.counts, w.prior, groups=w.groups, batch=w.batch, n_randomizations=100,
                                         return_posteriors=True, context=ctx)
    for lev, name in enumerate(["g1", "g2"]):
        ok, worst = _logp_close(res["joint.posteriors"][name].to_numpy(), fx[f"batch_jp{lev}"])
        assert ok, worst
    codes, bc = np.asarray(w.groups.codes), np.asarray(w.batch.codes)
    for lev in (0, 1):
        comp = np.bincount(bc[codes == lev], minlength=2).astype(np.int32)
        bj = api.scde_posteriors(w.models, w.counts, w.prior, n_randomizations=100, batch=w.batch, composition=comp,
                                 context=ctx)
        ok, worst = _logp_close(bj.to_numpy(), fx[f"batch_bjp{lev}"])
        assert ok, worst
    knn, counts = helpers.ref_knn_inputs()
    prior = pd.DataFrame({"x": np.linspace(0, 4.8, 401), "y": np.full(401, 1.0 / 401)})
    r = api.scde_posteriors(knn, counts, prior, n_randomizations=50, return_individual_posterior_modes=True, context=ctx)
    ok, worst = _logp_close(r["jp"].to_numpy(), fx["knn_jp"])
    assert ok, worst
    assert np.array_equal(r["modes"].to_numpy(), fx["knn_modes"])


def test_batch_models_and_na_batch_cells(ctx):
    """batch.models different from models (R/functions.R:304,356: the composition-sampled joints use their own error
    models) and NA entries in the batch factor (dropped from the pools and from the composition, as tapply / table do)
    against the oracle; the group joints must not change."""
    w = synth.make_workload(5, n_genes=90, n_cells=60, seed=17, batch=True)
    rng = np.random.default_rng(3)
    bm = w.models.copy()
    bm["corr.b"] = bm["corr.b"] + rng.uniform(-0.3, 0.3, len(bm))
    bm["conc.b"] = bm["conc.b"] - 0.5
    bcodes = np.asarray(w.batch.codes).copy()
    bcodes[[3, 17, 44]] = -1
    batch = pd.Categorical.from_codes(bcodes, categories=list(w.batch.categories))
    codes = np.asarray(w.groups.codes)
    want = O.expression_difference(w.models, w.counts, w.prior["x"].to_numpy(), w.prior["y"].to_numpy(),
                                   (np.nonzero(codes == 0)[0], np.nonzero(codes == 1)[0]), nboot=100, seed=1,
                                   batch_codes=bcodes, batch_models_df=bm)
    got = api.scde_expression_difference(w.models, w.counts, w.prior, groups=w.groups, batch=batch, batch_models=bm,
                                         n_randomizations=100, return_posteriors=True, context=ctx)
    for k, ref in (("results", want["results"]), ("batch.effect", want["batch.effect"]), ("batch.adjusted", want["batch.adjusted"])):
        _z_close(got[k]["Z"].to_numpy(), ref[:, 4])
        np.testing.assert_allclose(got[k][["lb", "mle", "ub"]].to_numpy(), ref[:, :3], rtol=1e-12, atol=1e-300)
    plain = api.scde_expression_difference(w.models, w.counts, w.prior, groups=w.groups, batch=batch, n_randomizations=100,
                                           context=ctx)
    assert np.array_equal(plain["results"].to_numpy(), got["results"].to_numpy())
    assert not np.array_equal(plain["batch.effect"]["Z"].to_numpy(), got["batch.effect"]["Z"].to_numpy())


def test_expression_prior_and_failure_probability_on_device(ctx):
    """scde.expression.prior / scde.failure.probability through the C ABI (csrc/prior.cu: magnitudes, weights, radix-select
    quantile and fixed-point BinDist on the device) against the oracle's restatement of R's density.default.  1e-9: the
    bins are 2^-62 fixed point (deterministic), the reference sums doubles sequentially."""
    from scde_b200 import prior as prior_mod

    cd = helpers.es_mef_raw()
    ifm = helpers.o_ifm()
    cd = cd[cd.sum(axis=1) > 0]
    cd = cd.loc[:, cd.sum(axis=0) > 1e4]
    ifm = ifm[ifm["corr.a"] > 0]
    cd = cd.loc[:, list(ifm.index)]
    for kw in (dict(), dict(max_quantile=0.999), dict(max_quantile=0.5), dict(max_value=5.0, bw=0.2, pseudo_count=3, length_out=250)):
        want = O.expression_prior(ifm, cd.to_numpy(), **kw)
        got = prior_mod.scde_expression_prior(ifm, cd, context=ctx, **kw)
        again = prior_mod.scde_expression_prior(ifm, cd, context=ctx, **kw)
        for k in ("x", "y", "lp", "grid.weight"):
            np.testing.assert_allclose(got[k].to_numpy(), want[k], rtol=1e-9, atol=1e-300, err_msg=f"{kw} {k}")
            assert np.array_equal(got[k].to_numpy(), again[k].to_numpy())  # integer bins: reproducible bit for bit
    # the prior the es.mef tests use (host twin, CPU fixtures) is the same prior
    _cd, _ifm, prior_host, _g = helpers.es_mef_inputs("tests")
    got = prior_mod.scde_expression_prior(ifm, cd, context=ctx)
    np.testing.assert_allclose(got["y"].to_numpy(), prior_host["y"].to_numpy(), rtol=1e-9)
    assert np.array_equal(got["x"].to_numpy(), prior_host["x"].to_numpy())
    # scde.failure.probability: counts form, magnitude-matrix form, common-vector form; 12-column models (conc.a2)
    sub = cd.iloc[:500]
    mag = O.expression_magnitude(sub.to_numpy(), ifm["corr.b"].to_numpy(), ifm["corr.a"].to_numpy())
    want = O.failure_probability(mag, ifm["conc.a"].to_numpy(), ifm["conc.b"].to_numpy())
    np.testing.assert_allclose(prior_mod.scde_failure_probability(ifm, counts=sub, context=ctx), want, rtol=1e-13, atol=1e-300)
    np.testing.assert_allclose(prior_mod.scde_failure_probability(ifm, magnitudes=mag, context=ctx), want, rtol=1e-13, atol=1e-300)
    knn = helpers.knn_models().iloc[:12]
    mags = np.array([1.0, 1.5, 2.0, -np.inf])
    m2 = np.repeat(mags[:, None], 12, axis=1)
    want = O.failure_probability(m2, knn["conc.a"].to_numpy(), knn["conc.b"].to_numpy(), knn["conc.a2"].to_numpy())
    np.testing.assert_allclose(prior_mod.scde_failure_probability(knn, magnitudes=mags, context=ctx), want, rtol=1e-13, atol=1e-300)


def test_r_shim_symbols_against_reference_fixtures(ctx):
    """integration/scde_b200_shim.cpp -- the file an scde maintainer puts into src/ in place of jpmatLogBoot.cpp and
    matSlideMult.cpp -- compiled against the header shim of the Rcpp API and driven through the same SEXP-building
    wrappers that drive the reference's own C++ (oracle/shim/ref_entry.cpp): .Call-shaped arguments -> shim ->
    libscde_b200.so, i.e. the code path of an R session minus R.  Compared with the reference fixtures / the oracle."""
    import ctypes
    import os

    from oracle import ref as R

    path = os.path.join(helpers.GOLD, "..", "..", "integration", "_build", "libscde_shim.so")
    if not os.path.exists(path):
        pytest.fail("integration/_build/libscde_shim.so is missing: __graft_entry__.build() builds it (make -C integration)")
    shim = ctypes.CDLL(os.path.abspath(path))
    keep, R._lib = R._lib, shim  # the oracle.ref binding, pointed at the shim build of the same five entry points
    try:
        fx = helpers.ref_fixtures()
        sub, ifm, prior, groups, sel = helpers.ref_cfg1_inputs()
        mm, lt, sq = O.pack_models(ifm)
        mag = O.marginals_from_prior_x(prior["x"].to_numpy())
        codes = np.asarray(groups.codes)
        jps = []
        for lev in (0, 1):
            ii = np.nonzero(codes == lev)[0]
            flat, off, uci = O.unique_counts(np.asfortranarray(sub.to_numpy()[:, ii]))
            r = R.log_boot_posterior(np.asfortranarray(mm[ii]), flat, off, uci, mag, 100, seed=1, returnpost=3)
            ok, worst = _logp_close(r["jp"], fx[f"cfg1_jp{lev}"])
            assert ok, worst
            assert np.array_equal(r["modes"], fx[f"cfg1_modes{lev}"])
            want = O.log_boot_posterior(np.asfortranarray(mm[ii]), flat, off, uci, mag, 100, seed=1, returnpost=2)["post"]
            for a, b in zip(r["post"], want):
                _rows_close(np.asarray(a), np.asarray(b))
            jps.append(fx[f"cfg1_jp{lev}"])
        py = prior["y"].to_numpy()
        assert np.array_equal(R.mat_slide_mult(jps[0] * py[None, :], jps[1] * py[None, :]), fx["cfg1_slide"])
        w = helpers.ref_batch_inputs()
        mm, lt, sq = O.pack_models(w.models)
        mag = O.marginals_from_prior_x(w.prior["x"].to_numpy())
        codes, bc = np.asarray(w.groups.codes), np.asarray(w.batch.codes)
        pools = [np.nonzero(bc == l)[0].astype(np.int32) for l in range(2)]
        flat, off, uci = O.unique_counts(w.counts)
        for lev in (0, 1):
            comp = np.bincount(bc[codes == lev], minlength=2).astype(np.int32)
            r = R.log_boot_batch_posterior(mm, flat, off, uci, mag, pools, comp, 100, seed=1, returnpost=1)
            ok, worst = _logp_close(r["jp"], fx[f"batch_bjp{lev}"])
            assert ok, worst
        rng = np.random.default_rng(11)
        matl = [np.asfortranarray(-rng.gamma(2.0, 3.0, size=(13, 29))) for _ in range(9)]
        np.testing.assert_allclose(R.jpmat_log_boot(matl, 40, seed=3), O.jpmat_log_boot(matl, 40, seed=3), rtol=1e-9)
        comp = np.array([3, 6], dtype=np.int32)
        np.testing.assert_allclose(R.jpmat_log_batch_boot([matl[:4], matl[4:]], comp, 25, seed=2),
                                   O.jpmat_log_batch_boot([matl[:4], matl[4:]], comp, 25, seed=2), rtol=1e-9)
    finally:
        R._lib = keep


def test_config2_posteriors_all_cells_and_magnitude(ctx):
    """BASELINE.json config 2: scde.posteriors(o.ifm, cd, o.prior) -- the joint posterior of ALL 40 es.mef.small cells as
    one group, every gene (13 788 x 40, tests/tests.R filter), 100 randomizations -- and scde.expression.magnitude on the
    same matrix, against the oracle (threaded over gene chunks with the Seed = 1 draws) and, for a spread gene sample
    with per-cell modes, against the oracle's full logBootPosterior."""
    cd, ifm, prior, groups = helpers.es_mef_inputs("tests")
    got = api.scde_posteriors(ifm, cd, prior, n_randomizations=100, context=ctx)
    assert got.shape == (cd.shape[0], 401)
    mm, lt, sq = O.pack_models(ifm)
    mag = O.marginals_from_prior_x(prior["x"].to_numpy())
    bi = O.boot_indices(1, len(ifm), 100)
    want = O.posteriors_chunked(mm, np.asfortranarray(cd.to_numpy()), mag, 100, bi, O.max_threads())
    ok, worst = _logp_close(got.to_numpy(), want)
    assert ok, worst
    np.testing.assert_allclose(got.to_numpy().sum(axis=1), 1.0, rtol=1e-12)
    sel = np.linspace(0, cd.shape[0] - 1, 48).astype(int)
    sub = cd.iloc[sel]
    r = api.scde_posteriors(ifm, sub, prior, n_randomizations=100, return_individual_posterior_modes=True, context=ctx)
    flat, off, uci = O.unique_counts(np.asfortranarray(sub.to_numpy()))
    w = O.log_boot_posterior(mm, flat, off, uci, mag, 100, seed=1, returnpost=1)
    ok, worst = _logp_close(r["jp"].to_numpy(), w["jp"])
    assert ok, worst
    assert np.array_equal(r["modes"].to_numpy(), w["modes"])
    ok, worst = _logp_close(r["jp"].to_numpy(), got.to_numpy()[sel])  # a gene's posterior does not depend on the other genes
    assert ok, worst
    m = api.scde_expression_magnitude(ifm, cd).to_numpy()
    wm = O.expression_magnitude(cd.to_numpy(), ifm["corr.b"].to_numpy(), ifm["corr.a"].to_numpy())
    fin = np.isfinite(wm)
    assert np.array_equal(np.isneginf(m), np.isneginf(wm))
    np.testing.assert_allclose(m[fin], wm[fin], rtol=1e-14, atol=1e-14)


def test_twin_batch_joints_equal_separate_launches(ctx):
    """the two composition-sampled joints of a batch-corrected call computed in one launch of the tcgen05 kernel (paired
    items on neighbouring SMs, scde_b200_options.twin_batch_joints) against one launch per joint: integer sums, so the
    results are bit-identical; 137 randomizations = two passes"""
    w = synth.make_workload(5, n_genes=333, n_cells=90, seed=23, batch=True)
    res = []
    for twin in (1, 0):
        keep = ctx.set_options(twin_batch_joints=twin)
        try:
            res.append(api.scde_expression_difference(w.models, w.counts, w.prior, groups=w.groups, batch=w.batch,
                                                      n_randomizations=137, return_posteriors=True, context=ctx))
        finally:
            ctx.restore_options(keep)
    for k in ("results", "batch.effect", "batch.adjusted"):
        assert np.array_equal(res[0][k].to_numpy(), res[1][k].to_numpy()), k
    assert np.array_equal(res[0]["batch.adjusted.difference.posterior"].to_numpy(),
                          res[1]["batch.adjusted.difference.posterior"].to_numpy())
    assert res[0]["stats"]["contract_cells"] == res[1]["stats"]["contract_cells"]
    # one launch per joint and pass: 4 joints x 2 passes; shared: the group joints pair their two passes (1 launch each), the
    # batch joints pair up per pass (2 launches)
    assert res[1]["stats"]["launches"]["contract"] == 8 and res[0]["stats"]["launches"]["contract"] == 4


@pytest.mark.parametrize("batch", [False, True])
def test_r_shim_fused_entry(ctx, batch):
    """`.Call("scde_b200_diff", ...)` of the R-package shim (integration/scde_b200_shim.cpp; what
    scde.expression.difference.b200 in integration/scde_b200.R calls) with .Call-shaped arguments: grid indices, Z and
    the BH-corrected cZ equal what the Python host layer gets from the same library call."""
    import ctypes
    import os

    path = os.path.abspath(os.path.join(helpers.GOLD, "..", "..", "integration", "_build", "libscde_shim.so"))
    if not os.path.exists(path):
        pytest.fail("integration/_build/libscde_shim.so is missing: __graft_entry__.build() builds it (make -C integration)")
    shim = ctypes.CDLL(path)
    w = synth.make_workload(5 if batch else 3, n_genes=120, n_cells=40, seed=29, batch=batch)
    mm, lt, sq = api.pack_models(w.models)
    x, y = w.prior["x"].to_numpy(), w.prior["y"].to_numpy()
    K, G, Cn = len(x), 120, 40
    counts = np.asfortranarray(w.counts, dtype=np.int32)
    group = np.asarray(w.groups.codes, dtype=np.int32)
    bc = np.asarray(w.batch.codes, dtype=np.int32) if batch else None
    n_sets = 3 if batch else 1
    idx, z, cz = np.zeros(n_sets * 3 * G), np.zeros(n_sets * G), np.zeros(n_sets * G)
    err = ctypes.create_string_buffer(256)
    dev = np.zeros(1, dtype=np.int32)
    dp, ip = ctypes.POINTER(ctypes.c_double), ctypes.POINTER(ctypes.c_int)
    rc = shim.shim_diff(counts.ctypes.data_as(ip), G, Cn, np.asfortranarray(mm).ctypes.data_as(dp), x.ctypes.data_as(dp),
                        y.ctypes.data_as(dp), K, group.ctypes.data_as(ip), bc.ctypes.data_as(ip) if batch else None,
                        2 if batch else 0, 100, K, 2 * K - 1, dev.ctypes.data_as(ip), 1, idx.ctypes.data_as(dp),
                        z.ctypes.data_as(dp), cz.ctypes.data_as(dp), err)
    assert rc == 0, err.value
    want = api.expression_difference_call(ctx, counts, mm, x, y, group, 100, 1, batch_codes=bc, n_batch_levels=2 if batch else 0,
                                          zero_index=[K], zero_index_adjusted=[2 * K - 1], local_theta=lt, sqlogit=sq)
    names = [("idx", "z", "cz")] + ([("batch_idx", "batch_z", "batch_cz"), ("adjusted_idx", "adjusted_z", "adjusted_cz")] if batch else [])
    for s, (ki, kz, kc) in enumerate(names):
        assert np.array_equal(idx[s * 3 * G:(s + 1) * 3 * G].reshape(3, G).T, want[ki])
        assert np.array_equal(z[s * G:(s + 1) * G], want[kz])
        assert np.array_equal(cz[s * G:(s + 1) * G], want[kc])
    # and cZ is the reference's: BH over all genes (oracle)
    pv = np.array([O.pnorm_upper(abs(v)) for v in want["z"]])
    adj = O.p_adjust_bh(pv)
    ref_cz = np.sign(want["z"]) * np.array([O.qnorm_upper(p) for p in adj])
    np.testing.assert_allclose(want["cz"], ref_cz, rtol=1e-9, atol=1e-12)
