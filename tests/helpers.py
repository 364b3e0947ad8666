"""Shared test inputs: the es.mef.small / o.ifm fixtures (tests/golden) prepared as tests/tests.R:8-38 does."""
from __future__ import annotations

import functools
import os

import numpy as np
import pandas as pd

GOLD = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")


@functools.lru_cache(maxsize=None)
def es_mef_raw():
    d = np.load(os.path.join(GOLD, "es_mef_small.npz"))
    return pd.DataFrame(d["counts"], index=[str(g) for g in d["genes"]], columns=[str(c) for c in d["cells"]])


@functools.lru_cache(maxsize=None)
def o_ifm():
    d = np.load(os.path.join(GOLD, "o_ifm.npz"))
    df = pd.DataFrame(d["values"], index=[str(c) for c in d["cells"]], columns=[str(c) for c in d["columns"]])
    df.attrs["groups"] = [str(g) for g in d["groups"]]
    return df


@functools.lru_cache(maxsize=None)
def knn_models():
    d = np.load(os.path.join(GOLD, "knn.npz"))
    return pd.DataFrame(d["values"], index=[str(c) for c in d["cells"]], columns=[str(c) for c in d["columns"]])


@functools.lru_cache(maxsize=None)
def es_mef_inputs(variant: str = "tests"):
    """(counts DataFrame, models DataFrame, prior DataFrame, groups Categorical).

    variant "tests":    the filter of tests/tests.R:19-21,33-38 (rowSums > 0, colSums > 1e4, corr.a > 0), default prior;
    variant "vignette": clean.counts(min.lib.size = 1000, min.reads = 1, min.detected = 1) and max.quantile = 0.999
                        -- the settings the printed vignette rows were produced with (SURVEY.md section 8(c)).
    """
    from prior_host import scde_expression_prior_host as scde_expression_prior
    from scde_b200.prior import clean_counts

    cd = es_mef_raw()
    ifm = o_ifm()
    if variant == "tests":
        cd = cd[cd.sum(axis=1) > 0]
        cd = cd.loc[:, cd.sum(axis=0) > 1e4]
        ifm = ifm[ifm["corr.a"] > 0]
        prior = scde_expression_prior(ifm, cd, length_out=400)
    else:
        cd = clean_counts(cd, min_lib_size=1000, min_reads=1, min_detected=1)
        ifm = ifm[ifm["corr.a"] > 0]
        prior = scde_expression_prior(ifm, cd, length_out=400, max_quantile=0.999)
    cd = cd.loc[:, list(ifm.index)]
    groups = pd.Categorical([("ESC" if n.startswith("ESC") else "MEF") for n in ifm.index], categories=["ESC", "MEF"])
    return cd, ifm, prior, groups


# ---- inputs of tests/golden/ref_fixtures_*.npz (outputs of the reference's own C++, tests/golden/make_ref_fixtures.py) ----
VIGNETTE_GENES = ["Dppa5a", "Pou5f1", "Gm13242", "Tdh", "Ift46", "4930509G22Rik"]


REF_FIXTURE_FILES = {"ref_fixtures_cfg1.npz": "cfg1_", "ref_fixtures_batch_knn.npz": ("batch_", "knn_")}


@functools.lru_cache(maxsize=None)
def ref_fixtures():
    """{name: array} of both fixture files (split by case so that each stays under 1 MB)"""
    out = {}
    for name in REF_FIXTURE_FILES:
        with np.load(os.path.join(GOLD, name)) as d:
            out.update({k: d[k] for k in d.files})
    return out


def ref_cfg1_inputs():
    """(counts of the selected genes, models, prior, groups, selected row numbers): 64 genes spread over the es.mef.small
    matrix (tests/tests.R filter) plus the six genes of vignettes/diffexp.md:113-119"""
    cd, ifm, prior, groups = es_mef_inputs("tests")
    names = list(cd.index)
    sel = sorted(set(np.linspace(0, len(names) - 1, 64).astype(int)) | {names.index(g) for g in VIGNETTE_GENES if g in names})
    return cd.iloc[sel], ifm, prior, groups, np.array(sel, dtype=np.int32)


def ref_knn_inputs():
    knn = knn_models().iloc[:12]
    rng = np.random.default_rng(3)
    counts = rng.negative_binomial(0.8, 0.02, size=(40, len(knn))).astype(np.int32)
    counts[rng.uniform(size=counts.shape) < 0.4] = 0
    return knn, np.asfortranarray(counts)


def ref_batch_inputs():
    from scde_b200 import synth

    return synth.make_workload(5, n_genes=48, n_cells=36, seed=3, batch=True)
