"""CPU tests that pin the oracle (oracle/scde_oracle.c): known answers for every third-party algorithm it restates,
the reference's printed vignette rows as an end-to-end smoke pin, and the committed golden output."""
import os

import mpmath as mp
import numpy as np
import pytest
from scipy.special import ndtri

import helpers
from oracle import oracle as O

mp.mp.dps = 50


def test_glibc_rand_known_answers():
    # SURVEY.md section 8(c)(i): srand(1) stream under the reference's rejection rule, glibc 2.39
    assert O.boot_indices(1, 20, 1)[0][:12].tolist() == [16, 7, 15, 15, 18, 3, 6, 15, 5, 11, 9, 12]
    assert O.boot_indices(1, 5000, 1)[0][:12].tolist() == [4200, 1971, 3915, 3992, 4558, 987, 1676, 3841, 1388, 2769,
                                                          2386, 3144]


def test_batch_boot_indices_stay_in_pools():
    pools = [np.array([0, 3, 4], np.int32), np.array([1, 2], np.int32), np.array([5], np.int32)]
    bi = O.batch_boot_indices(7, pools, [2, 0, 3], 50)
    assert bi.shape == (50, 5)
    assert np.isin(bi[:, :2], pools[0]).all() and (bi[:, 2:] == 5).all()


@pytest.mark.parametrize("x", [0, 1, 5, 627, 110329])
@pytest.mark.parametrize("theta", [0.01, 0.93, 1000.0])
@pytest.mark.parametrize("mu", [1e-3, 1.0, 1e4])
def test_dnbinom_against_mpmath(x, theta, mu):
    prob = theta / (theta + mu)
    p = mp.mpf(prob)
    th = mp.mpf(theta)
    exact = mp.loggamma(x + th) - mp.loggamma(th) - mp.loggamma(x + 1) + th * mp.log(p) + x * mp.log(1 - p)
    got = O.dnbinom_log(x, theta, prob)
    assert abs((got - exact) / exact) < 1e-12


def test_dnbinom_edge_cases():
    assert O.dnbinom_log(0, 0.7, 1.0) == 0.0            # mu = 0 at the first grid point
    assert O.dnbinom_log(3, 0.7, 1.0) == -np.inf
    assert np.isnan(O.dnbinom_log(3, 0.7, 0.0))


@pytest.mark.parametrize("x", [0, 1, 5, 627, 110329])
@pytest.mark.parametrize("lam", [0.1, 1.0, 1e4])
def test_dpois_against_mpmath(x, lam):
    exact = -mp.mpf(lam) + x * mp.log(mp.mpf(lam)) - mp.loggamma(x + 1)
    assert abs((O.dpois_log(x, lam) - exact) / exact) < 1e-13


def test_stirlerr_table_and_series():
    for i in range(1, 200):
        n = mp.mpf(i) / 2
        exact = mp.loggamma(n + 1) - (n + mp.mpf(1) / 2) * mp.log(n) + n - mp.log(mp.sqrt(2 * mp.pi))
        assert abs(O.stirlerr(i / 2) - exact) < 2e-16 + 1e-15 * abs(exact)


def test_qnorm_pnorm():
    for p in [1e-300, 4e-13, 1e-10, 1e-5, 0.01, 0.074, 0.076, 0.3, 0.5, 0.7, 0.93, 0.99, 1 - 1e-10]:
        want = -ndtri(p)
        assert abs(O.qnorm_upper(p) - want) <= 1e-14 * max(1.0, abs(want))
    assert O.qnorm_upper(0.0) == np.inf and O.qnorm_upper(1.0) == -np.inf
    for x in [0.0, 0.5, 3.0, 7.16, 20.0]:
        want = 0.5 * mp.erfc(mp.mpf(x) / mp.sqrt(2))
        assert abs(O.pnorm_upper(x) - want) / want < 1e-13


def test_slide_mult_is_full_cross_correlation():
    rng = np.random.default_rng(0)
    a, b = rng.random((5, 17)), rng.random((5, 17))
    got = O.mat_slide_mult(a, b)
    for g in range(5):
        np.testing.assert_allclose(got[g], np.correlate(a[g], b[g], "full"), rtol=1e-13)


def test_summary_hand_built_cases():
    n = 801
    diffv = O.fold_change_grid(np.linspace(0, 4.8, 401))
    P = np.zeros((4, n))
    P[0, 700:720] = 1 / 20     # all mass on the positive side -> Z saturates near +7.16
    P[1, 80:100] = 1 / 20      # all mass on the negative side
    P[2, :] = 1 / n            # flat: first maximum, symmetric
    P[3, 400] = 1.0            # point mass on zero
    res, idx = O.distribution_summary(P, diffv, 0.0)
    zmax = O.qnorm_upper(401e-15 / (1 + n * 1e-15))  # mass below + at H0 = 401 grid points of 1e-15
    assert abs(res[0, 4] - zmax) < 1e-9 and abs(res[1, 4] + zmax) < 5e-3
    assert idx[2, 1] == 0 and res[2, 4] == 0.0
    assert idx[0].tolist() == [699, 700, 719]  # lb = last point with cumulative mass < 2.5%
    assert idx[3].tolist() == [399, 400, 400] and res[3, 3] == 0.0
    # lb falls back to the first grid point when the first cumulative value already exceeds 2.5%
    P2 = np.zeros((1, n))
    P2[0, 0] = 0.5
    P2[0, n - 1] = 0.5
    res2, idx2 = O.distribution_summary(P2, diffv, 0.0)
    assert idx2[0].tolist() == [0, 0, n - 1]


def test_bh_matches_definition():
    rng = np.random.default_rng(5)
    p = rng.random(200)
    p[:5] = p[0]
    got = O.p_adjust_bh(p)
    o = np.argsort(-p, kind="stable")
    want = np.empty_like(p)
    want[o] = np.minimum(1, np.minimum.accumulate(len(p) / np.arange(len(p), 0, -1) * p[o]))
    np.testing.assert_allclose(got, want, rtol=1e-15)


def test_no_boot_equals_plain_product_and_modes():
    from scde_b200 import synth
    w = synth.make_workload(3, n_genes=30, n_cells=5, seed=2)
    mm, lt, sq = O.pack_models(w.models)
    mag = O.marginals_from_prior_x(w.prior["x"].to_numpy())
    flat, off, uci = O.unique_counts(w.counts)
    r = O.log_boot_posterior(mm, flat, off, uci, mag, 0, returnpost=3)
    lp = np.zeros((30, len(mag)))
    for c in range(5):
        tab, modes = O.cell_table(mm[c], flat[off[c]:off[c + 1]], mag, ncells_for_clamp=5)
        lp += tab.T[uci[:, c]]
        np.testing.assert_array_equal(r["modes"][:, c], mag[modes[uci[:, c]]])
    p = np.exp(lp - lp.max(axis=1, keepdims=True))
    np.testing.assert_allclose(r["jp"], p / p.sum(axis=1, keepdims=True), rtol=1e-12)


def _golden():
    d = np.load(os.path.join(helpers.GOLD, "es_mef_vignette_oracle.npz"))
    return d["results"], d["idx"], [str(g) for g in d["genes"]]


def test_vignette_smoke_pin():
    """The only golden numbers the reference holds for this path: six printed rows of vignettes/diffexp.md:113-119
    (a different libc rand() stream produced them, so this is a smoke pin with bootstrap-noise tolerances:
    Z within 0.05, bounds within 5 grid steps, at least five of the printed top six in the oracle's top six)."""
    res, idx, genes = _golden()
    vignette = {
        "Dppa5a": (8.075220, 9.984631, 11.575807, 8.075220, 7.160813),
        "Pou5f1": (5.370220, 7.200073, 9.189043, 5.370220, 7.160328),
        "Gm13242": (5.688455, 7.677425, 9.785734, 5.688455, 7.159979),
        "Tdh": (5.807793, 8.075220, 10.302866, 5.807793, 7.159589),
        "Ift46": (5.449779, 7.359190, 9.228822, 5.449779, 7.150242),
        "4930509G22Rik": (5.409999, 7.478528, 9.785734, 5.409999, 7.115605),
    }
    step = 0.0397793
    top6 = {genes[i] for i in np.argsort(-res[:, 4])[:6]}
    assert len(top6 & set(vignette)) >= 5
    for g, (lb, mle, ub, ce, z) in vignette.items():
        r = res[genes.index(g)]
        assert abs(r[4] - z) < 0.05
        assert abs(r[0] - lb) <= 5 * step + 1e-6 and abs(r[2] - ub) <= 5 * step + 1e-6 and abs(r[1] - mle) <= 5 * step + 1e-6
    dp = res[genes.index("Dppa5a")]
    assert abs(dp[0] - 8.075220) < 1e-6 and abs(dp[2] - 11.575807) < 1e-6 and abs(dp[4] - 7.160813) < 1e-6


def test_oracle_reproduces_committed_golden_slice():
    res, idx, genes = _golden()
    cd, ifm, prior, groups = helpers.es_mef_inputs("vignette")
    assert list(cd.index) == genes
    sel = np.r_[0:150, [genes.index("Dppa5a"), genes.index("Tdh")]]
    codes = np.asarray(groups.codes)
    out = O.expression_difference(ifm, cd.to_numpy()[sel], prior.x.to_numpy(), prior.y.to_numpy(),
                                  (np.nonzero(codes == 0)[0], np.nonzero(codes == 1)[0]), nboot=100, seed=1)
    np.testing.assert_allclose(out["results"][:, :5], res[sel, :5], rtol=1e-12, atol=1e-12)


def test_oracle_matches_reference_fixtures():
    """tests/golden/ref_fixtures_*.npz holds outputs of the reference's own C++ (src/jpmatLogBoot.cpp, src/matSlideMult.cpp
    compiled unmodified, tests/golden/make_ref_fixtures.py).  The oracle reproduces them BIT FOR BIT on config 1's data
    (es.mef.small + o.ifm, incl. the vignette's six genes), a batch case and the 12-column knn models -- this is what
    pins the oracle without the reference's sources (which the repository does not carry)."""
    fx = helpers.ref_fixtures()
    sub, ifm, prior, groups, sel = helpers.ref_cfg1_inputs()
    assert np.array_equal(sel, fx["cfg1_genes"])
    mm, lt, sq = O.pack_models(ifm)
    mag = O.marginals_from_prior_x(prior["x"].to_numpy())
    codes = np.asarray(groups.codes)
    jps = []
    for lev in (0, 1):
        ii = np.nonzero(codes == lev)[0]
        flat, off, uci = O.unique_counts(np.asfortranarray(sub.to_numpy()[:, ii]))
        r = O.log_boot_posterior(np.asfortranarray(mm[ii]), flat, off, uci, mag, 100, seed=1, returnpost=1)
        assert np.array_equal(r["jp"], fx[f"cfg1_jp{lev}"])
        assert np.array_equal(r["modes"], fx[f"cfg1_modes{lev}"])
        jps.append(r["jp"])
    py = prior["y"].to_numpy()
    assert np.array_equal(O.mat_slide_mult(jps[0] * py[None, :], jps[1] * py[None, :]), fx["cfg1_slide"])
    w = helpers.ref_batch_inputs()
    mm, lt, sq = O.pack_models(w.models)
    mag = O.marginals_from_prior_x(w.prior["x"].to_numpy())
    codes, bc = np.asarray(w.groups.codes), np.asarray(w.batch.codes)
    pools = [np.nonzero(bc == l)[0].astype(np.int32) for l in range(2)]
    flat_all, off_all, uci_all = O.unique_counts(w.counts)
    for lev in (0, 1):
        ii = np.nonzero(codes == lev)[0]
        flat, off, uci = O.unique_counts(np.asfortranarray(w.counts[:, ii]))
        assert np.array_equal(O.log_boot_posterior(np.asfortranarray(mm[ii]), flat, off, uci, mag, 100, seed=1)["jp"],
                              fx[f"batch_jp{lev}"])
        comp = np.bincount(bc[ii], minlength=2).astype(np.int32)
        assert np.array_equal(O.log_boot_batch_posterior(mm, flat_all, off_all, uci_all, mag, pools, comp, 100, seed=1)["jp"],
                              fx[f"batch_bjp{lev}"])
    knn, counts = helpers.ref_knn_inputs()
    mm, lt, sq = O.pack_models(knn)
    flat, off, uci = O.unique_counts(counts)
    r = O.log_boot_posterior(mm, flat, off, uci, O.marginals_from_prior_x(np.linspace(0, 4.8, 401)), 50, seed=1,
                             returnpost=1, localtheta=lt, sqlogit=sq)
    assert np.array_equal(r["jp"], fx["knn_jp"]) and np.array_equal(r["modes"], fx["knn_modes"])
