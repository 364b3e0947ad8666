"""CPU tests of the host logic and of the C-ABI library as far as it can go without a GPU."""
import ctypes as C
import os
import re

import numpy as np
import pandas as pd
import pytest

import helpers
from oracle import oracle as O
import prior_host as prior_mod
from scde_b200 import _lib, api, synth

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_library_loads_and_exports_every_declared_symbol():
    L = _lib.lib()
    header = open(os.path.join(ROOT, "include", "scde_b200.h")).read()
    declared = set(re.findall(r"SCDE_B200_API[^;]*?\b(scde_b200_\w+)\s*\(", header))
    assert declared == set(_lib.EXPORTED)
    for name in declared:
        assert hasattr(L, name), name
    assert L.scde_b200_version() == 100


def test_no_cpu_fallback_without_device():
    L = _lib.lib()
    if L.scde_b200_device_count() > 0:
        pytest.skip("a GPU is present")
    with pytest.raises(_lib.ScdeB200Error) as e:
        _lib.Context(0)
    assert e.value.code == -2 and "no CPU fallback" in str(e.value)


@pytest.mark.parametrize("seed,n,B", [(1, 20, 100), (1, 5000, 3), (12345, 7, 50), (0, 13, 10), (2, 1, 5), (77, 40, 150)])
def test_boot_indices_bit_exact_with_libc(seed, n, B):
    out = np.empty((B, n), np.int32)
    _lib.check(_lib.lib().scde_b200_boot_indices(seed, n, B, _lib.p_i32(out)))
    assert np.array_equal(out, O.boot_indices(seed, n, B))


def test_batch_boot_indices_bit_exact_with_libc():
    pools = [np.array([0, 3, 4, 9], np.int32), np.array([1, 2], np.int32), np.array([5, 6, 7, 8], np.int32)]
    off, cells = O.flatten_pools(pools)
    for comp in ([2, 0, 3], [4, 2, 4], [0, 0, 1]):
        comp = np.array(comp, np.int32)
        out = np.empty((30, int(comp.sum())), np.int32)
        _lib.check(_lib.lib().scde_b200_batch_boot_indices(9, 3, _lib.p_i32(off), _lib.p_i32(cells), _lib.p_i32(comp), 30,
                                                           _lib.p_i32(out)))
        assert np.array_equal(out, O.batch_boot_indices(9, pools, comp, 30))


def test_bh_cz_matches_oracle():
    rng = np.random.default_rng(1)
    z = np.r_[rng.normal(size=500) * 3, [7.160813, -7.160813, 0.0, 0.0]]
    cz = np.empty_like(z)
    _lib.check(_lib.lib().scde_b200_bh_cz(_lib.p_f64(z), len(z), _lib.p_f64(cz)))
    pa = O.p_adjust_bh(np.array([O.pnorm_upper(abs(v)) for v in z]))
    want = np.sign(z) * np.array([O.qnorm_upper(p) for p in pa])
    np.testing.assert_allclose(cz, want, rtol=1e-13, atol=1e-15)


def test_bh_cz_ties_and_degenerate_sizes():
    """long runs of saturated Z (equal p-values: the stable order decides nothing observable, the running minimum
    stays flat), all-equal input, n = 0 / 1 (R/functions.R:5051 on a one-gene data frame)"""
    rng = np.random.default_rng(2)
    z = rng.normal(size=3000) * 2.5
    z[::3], z[1::7], z[5::11] = 7.160813, -7.160813, 1e-9
    for zz in (z, np.full(17, 2.5), np.array([3.0]), np.empty(0)):
        zz = np.ascontiguousarray(zz, dtype=np.float64)
        cz = np.empty_like(zz)
        _lib.check(_lib.lib().scde_b200_bh_cz(_lib.p_f64(zz), len(zz), _lib.p_f64(cz)))
        if len(zz) == 0:
            continue
        pa = O.p_adjust_bh(np.array([O.pnorm_upper(abs(v)) for v in zz]))
        want = np.sign(zz) * np.array([O.qnorm_upper(p) for p in pa])
        np.testing.assert_allclose(cz, want, rtol=1e-13, atol=1e-15)
        assert (np.abs(cz) <= np.abs(zz) + 1e-12).all()  # the correction never makes a gene more significant


def test_fold_change_grid_and_zero_index():
    x = np.linspace(0, 4.8, 401)
    d = api.fold_change_grid(x)
    assert len(d) == 801 and d[0] == -4.8 and d[-1] == 4.8
    np.testing.assert_allclose(d, O.fold_change_grid(x), rtol=0, atol=1e-14)
    assert api._zero_index(d, 0.0).tolist() == [401]
    assert api._zero_index(d, [1.0, -2.0]).tolist() == [401 + round(np.log10(2) / 0.012), 401 - round(2 * np.log10(2) / 0.012)]


def test_pack_models_and_marginals():
    ifm = helpers.o_ifm().copy()
    ifm.iloc[3, ifm.columns.get_loc("corr.a")] = -0.2
    mm, lt, sq = api.pack_models(ifm)
    assert mm.shape == (40, 12) and lt == 0 and sq == 0 and mm[3, 4] == 1e-10 and np.isnan(mm[:, 6:]).all()
    mm2, lt2, sq2 = api.pack_models(helpers.knn_models())
    assert lt2 == 1 and sq2 == 1 and not np.isnan(mm2).any()
    m = api.marginals_from_prior(pd.DataFrame({"x": [0.0, 1.0, 2.0]}))
    assert m[0] == -np.inf and abs(m[1] - np.log(9)) < 1e-15


def test_unique_index_round_trip():
    w = synth.make_workload(3, n_genes=200, n_cells=7, seed=1)
    flat, off, uci = api._unique_index(w.counts)
    for c in range(7):
        assert np.array_equal(flat[off[c]:off[c + 1]][uci[:, c]], w.counts[:, c])
    f2, o2, u2 = O.unique_counts(w.counts)   # first-appearance order, same content
    for c in range(7):
        assert np.array_equal(f2[o2[c]:o2[c + 1]][u2[:, c]], w.counts[:, c])
        assert set(f2[o2[c]:o2[c + 1]]) == set(flat[off[c]:off[c + 1]])


def test_argument_validation_mirrors_reference():
    w = synth.make_workload(3, n_genes=10, n_cells=6, seed=1)
    with pytest.raises(ValueError, match="does not cover all of the cells"):
        api._counts_for_models(w.models, w.counts[:, :4])
    cd = pd.DataFrame(w.counts, columns=[f"x{i}" for i in range(6)])
    with pytest.raises(ValueError, match="does not cover all of the cells"):
        api._counts_for_models(w.models, cd)
    with pytest.raises(ValueError, match="composition must be provided"):
        api.scde_posteriors(w.models, w.counts, w.prior, batch=pd.Categorical(list("ababab")))


def test_expression_prior_shapes_match_survey_probes():
    cd, ifm, prior, groups = helpers.es_mef_inputs("tests")
    assert cd.shape == (13788, 40) and len(prior) == 401 and prior["x"].iloc[0] == 0.0
    assert abs(prior["x"].iloc[-1] - 8.69557) < 1e-4 and abs(prior["y"].sum() - 1) < 1e-12
    cd2, _, prior2, _ = helpers.es_mef_inputs("vignette")
    assert cd2.shape == (12142, 40) and abs(prior2["x"].iloc[-1] - 4.78992) < 1e-4


def test_density_restatement_against_exact_kde():
    rng = np.random.default_rng(0)
    x = rng.normal(size=4000)
    w = np.full(4000, 1 / 4000)
    gx, gy = prior_mod.density_gaussian(x, w, 0.1, 801, -3.0, 3.0)
    exact = np.array([np.sum(w * np.exp(-0.5 * ((g - x) / 0.1) ** 2)) / (0.1 * np.sqrt(2 * np.pi)) for g in gx])
    assert np.max(np.abs(gy - exact)) < 2e-3 * exact.max()


def test_synthetic_generator_is_deterministic():
    a = synth.make_workload(3, n_genes=50, n_cells=10)
    b = synth.make_workload(3, n_genes=50, n_cells=10)
    assert np.array_equal(a.counts, b.counts) and a.counts.flags["F_CONTIGUOUS"] and a.counts.dtype == np.int32
    assert 0.2 < (a.counts == 0).mean() < 0.8


def test_fisher_test_p_value():
    """fisher.test (R/functions.R:339): known answers -- R's documentation example (Agresti's tea tasting, p = 0.4857) and
    scipy's exact 2 x 2 routine; a 2 x 3 table goes through scipy's r x c code"""
    from scipy.stats import fisher_exact

    assert abs(api.fisher_test_p_value(np.array([[3, 1], [1, 3]])) - 0.4857142857142857) < 1e-12
    rng = np.random.default_rng(0)
    for _ in range(20):
        t = rng.integers(0, 40, size=(2, 2))
        if t.sum(axis=0).min() == 0 or t.sum(axis=1).min() == 0:
            continue
        assert abs(api.fisher_test_p_value(t) - fisher_exact(t).pvalue) < 1e-9
    assert 0.0 < api.fisher_test_p_value(np.array([[10, 3, 5], [4, 12, 7]])) < 0.1
    assert api.fisher_test_p_value(np.array([[5000, 0], [0, 5000]])) < 1e-300 or api.fisher_test_p_value(np.array([[5000, 0], [0, 5000]])) == 0.0


def test_strong_group_batch_interaction_warns(capsys, monkeypatch):
    """the reference prints a WARNING when groups and batches are confounded (p < 1e-3, R/functions.R:345-348); checked
    at the host layer with the device call stubbed out"""
    w = synth.make_workload(5, n_genes=4, n_cells=40, seed=2, batch=True)
    confounded = pd.Categorical(np.where(np.arange(40) < 20, "b1", "b2"))

    class Stop(Exception):
        pass

    def boom(*a, **k):
        raise Stop()

    monkeypatch.setattr(api, "expression_difference_call", boom)
    monkeypatch.setattr(api._lib, "default_context", lambda *a, **k: None)
    with pytest.raises(Stop):
        api.scde_expression_difference(w.models, w.counts, w.prior, groups=w.groups, batch=confounded)
    assert "strong interaction between groups and batches" in capsys.readouterr().out
    balanced = pd.Categorical(np.where(np.arange(40) % 2 == 0, "b1", "b2"))
    with pytest.raises(Stop):
        api.scde_expression_difference(w.models, w.counts, w.prior, groups=w.groups, batch=balanced)
    assert "strong interaction" not in capsys.readouterr().out


def test_prior_host_twin_against_oracle():
    """scde.expression.prior: the numpy twin (np.fft) against the oracle's C restatement of density.default (own radix-2
    FFT, BinDist, approx) on the es.mef.small data -- default, max.quantile = 0.999 (the vignette's setting) and explicit
    max.value / bw / pseudo.count"""
    cd = helpers.es_mef_raw()
    ifm = helpers.o_ifm()
    cd = cd[cd.sum(axis=1) > 0]
    cd = cd.loc[:, cd.sum(axis=0) > 1e4]
    ifm = ifm[ifm["corr.a"] > 0]
    cd = cd.loc[:, list(ifm.index)].iloc[::7]
    for kw in (dict(), dict(max_quantile=0.999), dict(max_value=5.0, bw=0.2, pseudo_count=3, length_out=250)):
        a = O.expression_prior(ifm, cd.to_numpy(), **kw)
        b = prior_mod.scde_expression_prior_host(ifm, cd, **kw)
        for k in ("x", "y", "lp", "grid.weight"):
            np.testing.assert_allclose(b[k].to_numpy(), a[k], rtol=1e-11, atol=1e-300)
